// nq_api.cu -- context, workspace, stage orchestration and the C ABI (include/nquant_b200.h).
// One translation unit: the stage kernels live in the .cuh files next to this one.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>
#include <utility>
#include <algorithm>
#include <mutex>
#include <thread>
#include <atomic>
#include <nvtx3/nvToolsExt.h>

#include "../../include/nquant_b200.h"
#include "nq_types.h"
#include "nq_math.h"
#include "nq_color.h"
#include "nq_bluenoise_table.h"
#include "nq_hist.cuh"
#include "nq_pnn.cuh"
#include "nq_dither.cuh"
#include "nq_dither_spec.cuh"

#define NQ_NSTAGES 6   // scan, histogram, find_nn sweep, merge, dither setup + saliency, dither
#define NQ_NKERNELS 4  // kernels timed on their own (nq_get_kernel_times): 0 k_spec_run, 1 k_dither_fifo, 2 k_dither_sorted, 3 k_merge_*

namespace {

thread_local std::string g_lastError;

int fail(int code, const std::string& msg) {
  g_lastError = msg;
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(NQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
  } while (0)

const signed char kBlueNoise[4096] = NQ_BLUE_NOISE_INIT;

// ---- generalized Hilbert order (GC:282-334, 356-365), explicit stack -----------------------------
struct GFrame { int x, y, ax, ay, bx, by; };
inline int sgn(int v) { return (v > 0) - (v < 0); }
template <class Emit>
void gilbert_walk(int width, int height, Emit emit) {
  std::vector<GFrame> st;
  st.reserve(256);
  if (width >= height) st.push_back({0, 0, width, 0, 0, height});
  else st.push_back({0, 0, 0, height, width, 0});
  while (!st.empty()) {
    GFrame f = st.back();
    st.pop_back();
    int x = f.x, y = f.y;
    const int ax = f.ax, ay = f.ay, bx = f.bx, by = f.by;
    const int w = abs(ax + ay), h = abs(bx + by);
    const int dax = sgn(ax), day = sgn(ay), dbx = sgn(bx), dby = sgn(by);
    if (h == 1) { for (int i = 0; i < w; ++i) { emit(x, y); x += dax; y += day; } continue; }
    if (w == 1) { for (int i = 0; i < h; ++i) { emit(x, y); x += dbx; y += dby; } continue; }
    int ax2 = ax / 2, ay2 = ay / 2, bx2 = bx / 2, by2 = by / 2;
    const int w2 = abs(ax2 + ay2), h2 = abs(bx2 + by2);
    if (2 * w > 3 * h) {
      if ((w2 % 2) != 0 && w > 2) { ax2 += dax; ay2 += day; }
      st.push_back({x + ax2, y + ay2, ax - ax2, ay - ay2, bx, by});   // visited second
      st.push_back({x, y, ax2, ay2, bx, by});                          // visited first
      continue;
    }
    if ((h2 % 2) != 0 && h > 2) { bx2 += dbx; by2 += dby; }
    st.push_back({x + (ax - dax) + (bx2 - dbx), y + (ay - day) + (by2 - dby), -bx2, -by2, -(ax - ax2), -(ay - ay2)});
    st.push_back({x + bx2, y + by2, ax, ay, bx - bx2, by - by2});
    st.push_back({x, y, bx2, by2, ax2, ay2});
  }
}

// ---- synthetic images (nquant_android_b200/synth.py) ---------------------------------------------
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__global__ void k_synth(uint32_t* out, int nimg, int width, int height, int cls, int amode, unsigned long long seed0) {
  const long long npix = (long long)width * height;
  const long long total = npix * nimg;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int img = (int)(g / npix);
    const long long idx = g - (long long)img * npix;
    const int x = (int)(idx % width), y = (int)(idx / width);
    const unsigned long long seed = seed0 + (unsigned long long)img;
    int v[3];
    const int bw = width - 1 > 1 ? width - 1 : 1, bh = height - 1 > 1 ? height - 1 : 1, bs = width + height - 2 > 1 ? width + height - 2 : 1;
    const int base[3] = {255 * x / bw, 255 * y / bh, 255 * (x + y) / bs};
    for (int ch = 0; ch < 3; ++ch) {
      unsigned long long h = mix64(seed ^ (((unsigned long long)idx * 4ULL + (unsigned long long)ch) * 0x9E3779B97F4A7C15ULL));
      if (cls == 2) v[ch] = (int)(h & 0xFF);
      else {
        const int amp = cls == 0 ? 2 : 32;
        int t = base[ch] + (int)(h % (unsigned long long)(2 * amp + 1)) - amp;
        v[ch] = t < 0 ? 0 : (t > 255 ? 255 : t);
      }
    }
    int a = 255;
    if (amode != 0) {
      if (amode == 2) a = 255 * (width - 1 - x) / bw;
      if (x < width / 8 && y < height / 8) a = 0;
    }
    out[g] = ((uint32_t)a << 24) | ((uint32_t)v[0] << 16) | ((uint32_t)v[1] << 8) | (uint32_t)v[2];
  }
}

__global__ void k_math_probe(int fn, const double* x, const double* y, double* out, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double r = 0;
  switch (fn) {
    case 0: r = nqm::nq_pow(x[i], y[i]); break;
    case 1: r = nqm::nq_exp(x[i]); break;
    case 2: r = nqm::nq_tanh(x[i]); break;
    case 3: r = nqm::nq_cbrt(x[i]); break;
    case 4: r = nqm::nq_atan2(x[i], y[i]); break;
    case 5: r = nqm::nq_sin(x[i]); break;
    case 6: r = nqm::nq_cos(x[i]); break;
  }
  out[i] = r;
}

__global__ void k_ciede_probe(const float* l1, const float* l2, float* out, int* nExact, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float L1 = l1[3 * i], A1 = l1[3 * i + 1], B1 = l1[3 * i + 2], L2 = l2[3 * i], A2 = l2[3 * i + 1], B2 = l2[3 * i + 2];
  nq::CiedeC cc;
  const float tL = nq::ciede_L(L1, L2);
  const float tC = nq::ciede_C(A1, B1, A2, B2, &cc);
  float tH, tRT;
  if (!nqf::ciede_HRT_fast(B1, B2, cc, tC, &tH, &tRT)) {
    double barC, barh;
    tH = nq::ciede_H(B1, B2, cc, &barC, &barh);
    tRT = nq::ciede_RT(barC, barh, tC, tH);
    atomicAdd(nExact, 1);
  }
  out[4 * i] = tL; out[4 * i + 1] = tC; out[4 * i + 2] = tH; out[4 * i + 3] = tRT;
}

__global__ void k_set_palette(NqImage* imgs, int img, const uint32_t* pal, int plen) {
  if (threadIdx.x < plen) imgs[img].palette[threadIdx.x] = pal[threadIdx.x];
  if (threadIdx.x == 0) imgs[img].paletteLen = plen;
}

// one RGB->Lab table per device, shared by every context on it
struct LabLutEntry { float4* ptr = nullptr; int refs = 0; };
std::mutex g_lutMutex;
std::map<int, LabLutEntry> g_lut;

struct DebugImage {
  std::vector<double> bins5;
  std::vector<float> initErr;
  std::vector<int> initNn;
  std::vector<int> merges;
  std::vector<float> sal;
};

}  // namespace

#define NQ_FRONT_STREAMS 2   // histogram / find_nn / merge of consecutive chunks alternate between these
#define NQ_SPEC_BULK_DEFAULT 0   // stage 6 record stream through cp.async.bulk + mbarrier (NQ_SPEC_BULK overrides)

struct nq_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;      // where the caller's order and timing live (nq_set_stream)
  cudaStream_t ownStream = nullptr;
  // internal streams of a call (convert_group): front = scan .. merge of a chunk, dith = dither of the chunks in order,
  // aux = the serial dither kernels next to the speculative rounds, copyOut / copyIn = device -> host of finished chunks and
  // host -> device of the coming ones
  cudaStream_t sFront[NQ_FRONT_STREAMS] = {}, sDith = nullptr, sAux = nullptr, sOut = nullptr, sIn = nullptr;
  std::vector<cudaEvent_t> evPool;    // grows on demand, reused by every call
  size_t evUsed = 0;
  int smCount = 148;
  // resident CTAs per SM of k_merge_lab<4>, k_merge_lab<8> and k_merge_rgb, from the occupancy calculator
  int mergeLab4PerSm = 0, mergeLab8PerSm = 0, mergeRgbPerSm = 0;
  unsigned long long launches = 0;
  bool debug = false;
  int chunkImages = 0;                // images per chunk (0 = automatic)
  // Gilbert orders by (w,h), least recently used first in orderLru
  std::map<std::pair<int, int>, uint32_t*> orders;
  std::vector<std::pair<int, int>> orderLru;
  size_t orderBytes = 0;
  // workspace
  unsigned char* ws = nullptr;
  size_t wsBytes = 0;
  NqImage* dImgs = nullptr;
  NqSlot* dSlots = nullptr;
  int* dLive = nullptr;
  int* dPos = nullptr;
  unsigned char* zeroPlane = nullptr;   // hCnt + hSum of every slot, contiguous: one memset per chunk
  unsigned char* memoPlane = nullptr;   // memo of every slot, contiguous
  unsigned char* sortPool = nullptr;    // NQ_FRONT_STREAMS x sortSets sets of CIELAB sort scratch
  size_t zeroSlotBytes = 0, memoSlotBytes = 0, sortSetBytes = 0, sortABytes = 0;
  int wsSlots = 0, wsNpix = 0, wsKind = -1, sortSets = 0;
  bool wsDebug = false, wsBits = false, wsIdx = false;
  std::vector<NqSlot> hSlots;
  // staging for host-buffer calls
  uint32_t* dIn = nullptr;
  uint32_t* dOut = nullptr;
  size_t stageBytes = 0;
  // per-stage device timing (CUDA events on the internal streams, summed over the chunks of a call)
  double stageMs[NQ_NSTAGES] = {};
  unsigned long long stageLaunches[NQ_NSTAGES] = {};
  // named kernels timed on their own (bench.py's roofline line): 0 = k_spec_run
  double kernelMs[NQ_NKERNELS] = {};
  unsigned long long kernelLaunches[NQ_NKERNELS] = {};
  // speculative segment-parallel dither (nq_dither_spec.cuh); on unless nq_set_spec_dither(0) / NQ_SPEC_DITHER=0
  bool specDither = true;
  int specSeg = 0, specWarm = 1024;
  size_t specPoolMaxBytes = 0;     // NQ_SPEC_POOL_GB: cap on the pool's memory (0 = 96 GB)
  int specSlotsMax = 0;            // cap on the pool of work-array slots (0 = none; NQ_SPEC_SLOTS, tests force slot reuse with it)
  nq::spec::SpecImage* dSpec = nullptr;
  int specCap = 0;                 // images dSpec holds
  unsigned char* specBuf = nullptr;
  size_t specBufBytes = 0;
  nq::spec::SpecWork* dSpecPool = nullptr;
  int* dSpecInts = nullptr;
  int specPoolCap = 0;
  float* dTanh = nullptr;          // (float) tanh(e / 255 * 20), e = -255 .. 255 (nq_dither_spec.cuh shape_tanh)
  unsigned long long specImages = 0, specRounds = 0, specFallbacks = 0;
  // results of the last batch
  std::vector<NqImage> lastImgs;
  std::vector<DebugImage> dbg;
};

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct SlotLayout {
  size_t keyOff, sal, bD, bF, bCnt, bErr, bNn, bTm, bMtm, heap, mergeLog, cells, bits, idx, total;
};
SlotLayout slot_layout(int kind, int npix, bool debug, bool needBits, bool needIdx) {
  SlotLayout L;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
  L.keyOff = take((NQ_NBINS + 1) * 4);
  const bool lab = kind == NQ_KIND_LAB;
  L.sal = take(lab && debug ? (size_t)npix * 4 : 0);  // the dither kernel derives saliency itself; kept for parity tests
  L.bD = take((size_t)4 * NQ_NBINS * 8);
  L.bF = take((size_t)4 * NQ_NBINS * 4);
  L.bCnt = take(NQ_NBINS * 4);
  L.bErr = take(NQ_NBINS * 4);
  L.bNn = take(NQ_NBINS * 4);
  L.bTm = take(NQ_NBINS * 4);
  L.bMtm = take(NQ_NBINS * 4);
  L.heap = take((NQ_NBINS + 2) * 8);
  L.mergeLog = take(debug ? (size_t)2 * NQ_NBINS * 4 : 0);
  L.cells = take(lab ? (size_t)32768 * 32 : 0);
  L.bits = take(needBits ? ((size_t)1 << 29) : 0);      // one bit per ARGB value
  L.idx = take(needIdx ? (size_t)npix * 2 : 0);         // first-pass indices + pending marks of the per-pixel BlueNoise pass
  L.total = o;
  return L;
}

// Sort scratch of the strict-order CIELAB histogram (2 x npix words + run counters per image) is only
// needed while an image's histogram is being built, so a small pool of sets is cycled through the
// batch instead of giving every image its own. Every front stream owns NQ_SORT_POOL of them.
#define NQ_SORT_POOL 32

int ensure_workspace(nq_ctx* c, int kind, int npix, int wantSlots, bool needBits, bool needIdx) {
  SlotLayout L = slot_layout(kind, npix, c->debug, needBits, needIdx);
  const bool lab = kind == NQ_KIND_LAB;
  const size_t nruns = ((size_t)npix + NQ_RUN - 1) / NQ_RUN;
  const size_t sortA = align_up((size_t)npix * 4, 256);
  const size_t sortSet = lab ? sortA * 2 + align_up(nruns * 256 * 4, 256) : 0;
  const size_t zeroSlot = (size_t)NQ_NBINS * 4 + (size_t)4 * NQ_NBINS * 8, memoSlot = (size_t)NQ_NBINS * 2;
  size_t freeB = 0, totalB = 0;
  CU(cudaMemGetInfo(&freeB, &totalB));
  const size_t budget = (size_t)((double)(freeB + c->wsBytes) * 0.85);
  const size_t perImage = L.total + zeroSlot + memoSlot + sizeof(NqImage) + sizeof(NqSlot) + 2 * NQ_NBINS * 4 + 1024;
  int pool = std::min(wantSlots, NQ_SORT_POOL);
  while (pool > 1 && NQ_FRONT_STREAMS * pool * sortSet + perImage > budget) pool /= 2;
  if (NQ_FRONT_STREAMS * pool * sortSet + perImage > budget) return fail(NQ_ERR_NOMEM, "not enough device memory for one image workspace");
  const int maxSlots = (int)std::min<size_t>((budget - NQ_FRONT_STREAMS * pool * sortSet) / perImage, 8192);
  const int slots = std::min(wantSlots, maxSlots);
  if (c->ws && c->wsKind == kind && c->wsNpix == npix && c->wsSlots >= slots && c->wsDebug == c->debug && c->wsBits == needBits && c->wsIdx == needIdx) return NQ_OK;
  if (c->ws) { CU(cudaDeviceSynchronize()); cudaFree(c->ws); c->ws = nullptr; c->wsBytes = 0; c->wsSlots = 0; }
  const size_t imgsB = align_up(sizeof(NqImage) * slots, 256), slotsB = align_up(sizeof(NqSlot) * slots, 256);
  const size_t liveB = align_up((size_t)slots * NQ_NBINS * 4, 256);
  const size_t total = imgsB + slotsB + 2 * liveB + (zeroSlot + memoSlot + L.total) * slots + sortSet * pool * NQ_FRONT_STREAMS;
  CU(cudaMalloc(&c->ws, total));
  c->wsBytes = total;
  unsigned char* p = c->ws;
  c->dImgs = reinterpret_cast<NqImage*>(p); p += imgsB;
  c->dSlots = reinterpret_cast<NqSlot*>(p); p += slotsB;
  c->dLive = reinterpret_cast<int*>(p); p += liveB;
  c->dPos = reinterpret_cast<int*>(p); p += liveB;
  c->zeroPlane = p; p += zeroSlot * slots;
  c->memoPlane = p; p += memoSlot * slots;
  c->sortPool = p; p += sortSet * pool * NQ_FRONT_STREAMS;
  c->zeroSlotBytes = zeroSlot; c->memoSlotBytes = memoSlot; c->sortSetBytes = sortSet; c->sortABytes = sortA;
  c->hSlots.assign(slots, NqSlot{});
  for (int s = 0; s < slots; ++s) {
    unsigned char* b = p + L.total * s;
    NqSlot& S = c->hSlots[s];
    S.hCnt = reinterpret_cast<unsigned int*>(c->zeroPlane + zeroSlot * s);
    S.hSum = reinterpret_cast<unsigned long long*>(c->zeroPlane + zeroSlot * s + (size_t)NQ_NBINS * 4);
    S.keyOff = reinterpret_cast<unsigned int*>(b + L.keyOff);
    S.sal = (lab && c->debug) ? reinterpret_cast<float*>(b + L.sal) : nullptr;
    double* bd = reinterpret_cast<double*>(b + L.bD);
    S.bAc = bd; S.bC1 = bd + NQ_NBINS; S.bC2 = bd + 2 * NQ_NBINS; S.bC3 = bd + 3 * NQ_NBINS;
    float* bf = reinterpret_cast<float*>(b + L.bF);
    S.fAc = bf; S.fC1 = bf + NQ_NBINS; S.fC2 = bf + 2 * NQ_NBINS; S.fC3 = bf + 3 * NQ_NBINS;
    S.bCnt = reinterpret_cast<float*>(b + L.bCnt);
    S.bErr = reinterpret_cast<float*>(b + L.bErr);
    S.bNn = reinterpret_cast<int*>(b + L.bNn);
    S.bTm = reinterpret_cast<int*>(b + L.bTm);
    S.bMtm = reinterpret_cast<int*>(b + L.bMtm);
    S.heap = reinterpret_cast<uint2*>(b + L.heap);
    S.mergeLog = c->debug ? reinterpret_cast<int*>(b + L.mergeLog) : nullptr;
    S.memo = reinterpret_cast<unsigned short*>(c->memoPlane + memoSlot * s);
    S.cells = lab ? b + L.cells : nullptr;
    S.bits = needBits ? reinterpret_cast<unsigned int*>(b + L.bits) : nullptr;
    S.idx = needIdx ? reinterpret_cast<unsigned short*>(b + L.idx) : nullptr;
  }
  c->wsSlots = slots; c->wsNpix = npix; c->wsKind = kind; c->sortSets = pool; c->wsDebug = c->debug; c->wsBits = needBits; c->wsIdx = needIdx;
  return NQ_OK;
}

// The visiting order of a (w, h) image is a table of 4 bytes per pixel, built by a host walk the first time the size is
// seen. The cache is bounded (entries and bytes): a long-lived context that serves many sizes evicts the least recently used.
#define NQ_ORDER_MAX_ENTRIES 8
#define NQ_ORDER_MAX_BYTES ((size_t)2 << 30)
int ensure_order(nq_ctx* c, int w, int h, const uint32_t** out) {
  auto key = std::make_pair(w, h);
  auto it = c->orders.find(key);
  if (it != c->orders.end()) {
    auto pos = std::find(c->orderLru.begin(), c->orderLru.end(), key);
    if (pos != c->orderLru.end()) { c->orderLru.erase(pos); c->orderLru.push_back(key); }
    *out = it->second;
    return NQ_OK;
  }
  if (w > 65535 || h > 65535) return fail(NQ_ERR_ARG, "image side exceeds 65535");
  const size_t bytes = (size_t)w * h * 4;
  while (!c->orderLru.empty() && (c->orderLru.size() >= NQ_ORDER_MAX_ENTRIES || c->orderBytes + bytes > NQ_ORDER_MAX_BYTES)) {
    const auto old = c->orderLru.front();
    c->orderLru.erase(c->orderLru.begin());
    CU(cudaDeviceSynchronize());                    // nothing in flight may still read the table
    cudaFree(c->orders[old]);
    c->orderBytes -= (size_t)old.first * old.second * 4;
    c->orders.erase(old);
  }
  std::vector<uint32_t> host;
  host.reserve((size_t)w * h);
  gilbert_walk(w, h, [&](int x, int y) { host.push_back((uint32_t)x | ((uint32_t)y << 16)); });
  if (host.size() != (size_t)w * h) return fail(NQ_ERR_ARG, "gilbert walk size mismatch");
  uint32_t* d = nullptr;
  CU(cudaMalloc(&d, bytes));
  cudaError_t e = cudaMemcpy(d, host.data(), bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(d); return fail(NQ_ERR_CUDA, std::string("cudaMemcpy(order): ") + cudaGetErrorString(e)); }
  c->orders[key] = d;
  c->orderLru.push_back(key);
  c->orderBytes += bytes;
  *out = d;
  return NQ_OK;
}

int pixel_grid_x(const nq_ctx* c, int npix, int nimg) {
  int want = (npix + 256 * 8 - 1) / (256 * 8);
  int cap = std::max(1, (c->smCount * 8) / std::max(1, nimg));
  return std::max(1, std::min(want, cap));
}

cudaEvent_t take_event(nq_ctx* c) {
  if (c->evUsed == c->evPool.size()) {
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    c->evPool.push_back(e);
  }
  return c->evPool[c->evUsed++];
}

struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// One chunk of a call: images [base, base + n) of the group, with the events that bracket its stages.
struct Chunk {
  int base = 0, n = 0;
  int mergeInFlight = 0;           // images whose merge loops can run next to each other: this chunk's and a neighbour's
  cudaStream_t front = nullptr;
  int frontIdx = 0;
  cudaEvent_t evIn = nullptr;      // host-buffer calls: the chunk's pixels have arrived (copy-in stream)
  cudaEvent_t ev[5] = {};          // on `front`: start, after scan, after histogram, after the find_nn sweep, after the merge loop
  cudaEvent_t evD[3] = {};         // on the dither stream: start, after setup, end
  cudaEvent_t evK[2 * NQ_NKERNELS] = {};   // pairs around the kernels timed on their own (0 when not recorded)
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> evRuns;   // around every k_spec_run launch
  unsigned long long launches[NQ_NSTAGES] = {};
  // host-buffer calls: images [0, copied) of the chunk are already on their way to the host (progressive copy-out)
  int copied = 0;
  uint32_t* hOut = nullptr;        // host destination of the chunk's first image, or nullptr
  const uint32_t* dOut = nullptr;  // device source of the chunk's first image
  size_t imageBytes = 0;
};

// launches and small copies of the admission / round loop (spec_drive in nq_dither_spec.cuh) on the dither stream
struct SpecCudaBackend {
  nq_ctx* c;
  Chunk* ch;
  cudaStream_t st;
  bool timing = false;
  cudaEvent_t t0 = nullptr, t1 = nullptr;
  cudaError_t err = cudaSuccess;
  template <class... P, class... A>
  void launch(void (*kernel)(P...), dim3 grid, int block, A... args) {
    kernel<<<grid, block, 0, st>>>(args...);
    ++c->launches;
  }
  // stage 6 (k_spec_run): bracketed by its own events, for nq_get_kernel_times
  template <class... P, class... A>
  void launch_run(void (*kernel)(P...), dim3 grid, int block, A... args) {
    cudaEvent_t a = take_event(c), b = take_event(c);
    cudaEventRecord(a, st);
    kernel<<<grid, block, 0, st>>>(args...);
    cudaEventRecord(b, st);
    ch->evRuns.emplace_back(a, b);
    ++c->launches;
  }
  void keep(cudaError_t e) { if (err == cudaSuccess && e != cudaSuccess) err = e; }
  void write_ints(int* dev, const int* host, int n) { keep(cudaMemcpyAsync(dev, host, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st)); }
  void read_ints(int* host, const int* dev, int n) {
    keep(cudaMemcpyAsync(host, dev, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    keep(cudaStreamSynchronize(st));
  }
  // NQ_SPEC_TIMING=1: device time of every launch of this path on stderr (synchronises after each; diagnosis only)
  void begin() { if (timing) { cudaEventCreate(&t0); cudaEventCreate(&t1); cudaEventRecord(t0, st); } }
  void end() { if (timing) { cudaEventDestroy(t0); cudaEventDestroy(t1); } }
  void lap(const char* what) {
    if (!timing) return;
    cudaEventRecord(t1, st);
    cudaEventSynchronize(t1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, t0, t1);
    fprintf(stderr, "[nq spec] %-14s %9.3f ms\n", what, ms);
    cudaEventRecord(t0, st);
  }
  // images [0, prefix) of the chunk are complete: copy them out on the copy-out stream while the rest is still being dithered
  void done_prefix(int prefix) {
    if (!ch->hOut || prefix - ch->copied < 16) return;
    cudaEvent_t e = take_event(c);
    keep(cudaEventRecord(e, st));
    keep(cudaStreamWaitEvent(c->sOut, e, 0));
    keep(cudaMemcpyAsync(ch->hOut + (size_t)ch->copied * (ch->imageBytes / 4), ch->dOut + (size_t)ch->copied * (ch->imageBytes / 4),
                         (size_t)(prefix - ch->copied) * ch->imageBytes, cudaMemcpyDeviceToHost, c->sOut));
    ch->copied = prefix;
  }
  void note(int round, int active, int open, int patches, int redos) {
    if (timing) fprintf(stderr, "[nq spec] round %d: %d image(s) in the pool, %d open, %d patch(es), %d re-resolve(s)\n", round, active, open, patches, redos);
  }
};

// Speculative segment-parallel dither of the chunk's images that qualify, on stream `st`, in two steps so that the
// serial kernels of the other images can be enqueued in between. spec_prepare: the pool of work-array slots and
// k_spec_setup, which decides on the device which images are taken (NqImage::specDone = 2, elig[i] = 1) -- synchronises.
// spec_rounds: the admission / round loop; images it completes get specDone = 1, images it took but could not finish 3
// (listed in `handed`).
struct SpecPlan { int seg = 0, nslots = 0, any = 0; };
int spec_prepare(nq_ctx* c, Chunk& ch, cudaStream_t st, int npix, const uint32_t* dOrder, std::vector<int>& elig, SpecPlan* plan) {
  using namespace nq::spec;
  const int n = ch.n;
  elig.assign(n, 0);
  *plan = SpecPlan{};
  int seg = c->specSeg;
  const int warm = c->specWarm;
  if (seg == 0) {   // automatic: 8192-pixel segments when that gives the machine enough threads, shorter ones for small jobs
    const long long total = (long long)n * (long long)npix;
    seg = total / 8192 >= 32768 ? 8192 : (int)std::max<long long>(2048, (total / 32768 + 255) / 256 * 256);
    if (seg > 8192) seg = 8192;
  }
  if (npix < 4 * seg) return NQ_OK;
  const int nTotal = c->wsSlots;
  if (c->specCap < nTotal) {
    if (c->dSpec) { CU(cudaDeviceSynchronize()); cudaFree(c->dSpec); }
    c->dSpec = nullptr; c->specCap = 0;
    CU(cudaMalloc(&c->dSpec, sizeof(SpecImage) * (size_t)nTotal));
    c->specCap = nTotal;
  }
  const SpecLayout L = spec_layout(npix, seg);
  size_t freeB = 0, totalB = 0;
  CU(cudaMemGetInfo(&freeB, &totalB));
  // The rounds are latency bound (a round lasts as long as its slowest thread: a chain of segments run sequentially), so the
  // throughput of the path is images in the pool / (rounds per image x round time): the pool takes up to 300 4K images
  // (one thread per segment: the SMs filled four times over) and up to half of the free memory, at most 96 GB.
  const size_t poolCap = c->specPoolMaxBytes ? c->specPoolMaxBytes : ((size_t)96 << 30);
  const size_t budget = std::min<size_t>((size_t)((double)(freeB + c->specBufBytes) * 0.5), poolCap);
  const long long wantThreads = (long long)c->smCount * 2048;
  int nslots = (int)std::min<long long>(n, std::max<long long>(8, (wantThreads + L.nseg - 1) / L.nseg));
  nslots = (int)std::min<size_t>((size_t)nslots, budget / L.perSlot);
  if (c->specSlotsMax > 0) nslots = std::min(nslots, c->specSlotsMax);
  if (nslots < 1) return NQ_OK;                     // no room: the serial kernel does the work
  if (c->specBufBytes < L.perSlot * (size_t)nslots) {
    if (c->specBuf) { CU(cudaDeviceSynchronize()); cudaFree(c->specBuf); }
    c->specBuf = nullptr; c->specBufBytes = 0;
    CU(cudaMalloc(&c->specBuf, L.perSlot * (size_t)nslots));
    c->specBufBytes = L.perSlot * (size_t)nslots;
  }
  if (c->specPoolCap < nslots) {
    if (c->dSpecPool) { CU(cudaDeviceSynchronize()); cudaFree(c->dSpecPool); cudaFree(c->dSpecInts); }
    c->dSpecPool = nullptr; c->dSpecInts = nullptr; c->specPoolCap = 0;
    CU(cudaMalloc(&c->dSpecPool, sizeof(SpecWork) * (size_t)nslots));
    CU(cudaMalloc(&c->dSpecInts, sizeof(int) * (size_t)(4 * nslots + 4)));
    c->specPoolCap = nslots;
  }
  std::vector<SpecWork> pool(nslots);
  spec_bind_pool(pool.data(), nslots, c->specBuf, L);
  CU(cudaMemcpyAsync(c->dSpecPool, pool.data(), sizeof(SpecWork) * (size_t)nslots, cudaMemcpyHostToDevice, st));
  int* dElig = reinterpret_cast<int*>(c->specBuf);      // scratch: the pool's work arrays are not in use yet
  k_spec_setup<<<(n + 63) / 64, 64, 0, st>>>(c->dImgs + ch.base, c->dSlots + ch.base, c->dSpec + ch.base, dOrder, n, seg, warm, dElig); ++c->launches;
  CU(cudaMemcpyAsync(elig.data(), dElig, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));                    // also keeps `pool` alive until the copy is done
  for (int i = 0; i < n; ++i) plan->any += (elig[i] & 255) == 1;
  plan->seg = seg; plan->nslots = nslots;
  return NQ_OK;
}
int spec_rounds(nq_ctx* c, Chunk& ch, cudaStream_t st, int npix, const SpecPlan& plan, const std::vector<int>& elig, std::vector<int>& handed) {
  using namespace nq::spec;
  handed.clear();
  if (!plan.any) return NQ_OK;
  SpecCudaBackend be{c, &ch, st};
  be.timing = getenv("NQ_SPEC_TIMING") != nullptr;
  be.begin();
  SpecStats stats;
  handed.assign(plan.any, 0);
  spec_drive(be, c->dImgs + ch.base, c->dSpec + ch.base, c->dSpecPool, elig.data(), ch.n, npix, plan.seg, plan.nslots, c->dSpecInts, c->dTanh,
             c->smCount, &stats, handed.data());
  handed.resize((size_t)stats.handedBack);
  be.end();
  c->specImages += stats.done; c->specRounds += stats.rounds; c->specFallbacks += stats.handedBack;
  CU(be.err);
  CU(cudaGetLastError());
  return NQ_OK;
}

struct GroupArgs {
  int kind, w, h, nmax, dither;
  const uint64_t* seeds;
  const uint32_t* dPalIn;
  int palInLen;
  const uint32_t* hIn;     // host pixels (nullptr: dIn is the caller's device buffer and already holds them)
  uint32_t* hOut;
  bool stopAfterSweep = false;   // stage hook nq_histogram: no merge loop, no dither
};

// Instance of k_merge_lab for a chunk: the one with 4 CTAs per SM has the shorter chain per image and is used while the merge
// loops that can run at once (this chunk's and the other front stream's) fit one wave of it; beyond that, the one with 8.
int lab_merge_ctas(const nq_ctx* c, const Chunk& ch) { return ch.mergeInFlight > c->smCount * c->mergeLab4PerSm ? 8 : 4; }

// scan .. merge loop of one chunk, enqueued on its front stream (no host synchronisation unless the context is in debug mode)
int enqueue_front(nq_ctx* c, Chunk& ch, const GroupArgs& A, const uint32_t* dIn, uint32_t* dOut) {
  NvtxRange nv("nq front (scan, histogram, find_nn, merge)");
  const int n = ch.n, npix = A.w * A.h, kind = A.kind, nmax = A.nmax;
  cudaStream_t st = ch.front;
  NqImage* dI = c->dImgs + ch.base;
  NqSlot* dS = c->dSlots + ch.base;
  if (ch.evIn) CU(cudaStreamWaitEvent(st, ch.evIn, 0));
  std::vector<NqImage> hImgs(n);
  for (int i = 0; i < n; ++i) {
    NqImage& I = hImgs[i];
    memset(&I, 0, sizeof(I));
    I.kind = kind; I.width = A.w; I.height = A.h; I.npix = npix; I.nmax = nmax; I.dither = A.dither;
    I.seed = A.seeds ? A.seeds[ch.base + i] : 0ULL;
    I.transIdx = -1;
    I.mergeCtas = kind == NQ_KIND_LAB ? (lab_merge_ctas(c, ch) == 8 ? c->mergeLab8PerSm : c->mergeLab4PerSm) : c->mergeRgbPerSm;
    NqSlot& S = c->hSlots[ch.base + i];
    S.in = dIn + (size_t)(ch.base + i) * npix;
    S.out = dOut + (size_t)(ch.base + i) * npix;
    if (kind == NQ_KIND_LAB) {   // sort scratch: the sets of this chunk's front stream, cycled through the chunk
      unsigned char* sp = c->sortPool + c->sortSetBytes * ((size_t)ch.frontIdx * c->sortSets + (size_t)(i % c->sortSets));
      S.sortA = reinterpret_cast<uint32_t*>(sp);
      S.sortB = reinterpret_cast<uint32_t*>(sp + c->sortABytes);
      S.warpHist = reinterpret_cast<unsigned int*>(sp + 2 * c->sortABytes);
    }
  }
  CU(cudaMemcpyAsync(dI, hImgs.data(), sizeof(NqImage) * n, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(dS, c->hSlots.data() + ch.base, sizeof(NqSlot) * n, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(c->zeroPlane + c->zeroSlotBytes * ch.base, 0, c->zeroSlotBytes * n, st));
  CU(cudaMemsetAsync(c->memoPlane + c->memoSlotBytes * ch.base, 0xFF, c->memoSlotBytes * n, st));
  for (int i = 0; i < n; ++i) if (c->hSlots[ch.base + i].bits) CU(cudaMemsetAsync(c->hSlots[ch.base + i].bits, 0, (size_t)1 << 29, st));
  const int gx = pixel_grid_x(c, npix, n);
  const dim3 pg(gx, n);
  unsigned long long l0 = c->launches;
  auto mark = [&](int k) { cudaEventRecord(ch.ev[k], st); if (k > 0) { ch.launches[k - 1] += c->launches - l0; l0 = c->launches; } };
  mark(0);
  nq::k_alpha_scan<<<pg, 256, 0, st>>>(dI, dS); ++c->launches;
  nq::k_setup_scan<<<(n + 127) / 128, 128, 0, st>>>(dI, dS, n); ++c->launches;
  mark(1);
  if (nmax > 2) {
    if (kind == NQ_KIND_RGB) {
      {  // contiguous tiles per CTA; enough CTAs to fill the machine twice over
        const int ntiles = ((A.w + NQ_HTW - 1) / NQ_HTW) * ((A.h + NQ_HTW - 1) / NQ_HTW);
        const dim3 hg(std::max(1, std::min(ntiles, std::max(1, c->smCount * 8 / n))), n);
        nq::k_hist_rgb<<<hg, 256, sizeof(nq::HistTable), st>>>(dI, dS); ++c->launches;
      }
      nq::k_finalize_rgb<<<n, 1024, 0, st>>>(dI, dS); ++c->launches;
    } else {
      const int nruns = (npix + NQ_RUN - 1) / NQ_RUN;
      nq::k_lab_count<<<pg, 256, 0, st>>>(dI, dS); ++c->launches;
      nq::k_lab_scan_keys<<<n, 1024, 0, st>>>(dI, dS); ++c->launches;
      for (int g0 = 0; g0 < n; g0 += c->sortSets) {   // images of one group own distinct sort scratch sets
        const int gn = std::min(c->sortSets, n - g0);
        NqImage* gi = dI + g0;
        NqSlot* gs = dS + g0;
        const dim3 rg(std::max(1, std::min((nruns + 7) / 8, std::max(1, c->smCount * 8 / gn))), gn);
        nq::k_radix_count<0><<<rg, 256, 0, st>>>(gi, gs); ++c->launches;
        nq::k_radix_offsets<<<gn, 256, 0, st>>>(gi, gs); ++c->launches;
        nq::k_radix_scatter<0><<<rg, 256, 0, st>>>(gi, gs); ++c->launches;
        nq::k_radix_count<1><<<rg, 256, 0, st>>>(gi, gs); ++c->launches;
        nq::k_radix_offsets<<<gn, 256, 0, st>>>(gi, gs); ++c->launches;
        nq::k_radix_scatter<1><<<rg, 256, 0, st>>>(gi, gs); ++c->launches;
        const dim3 bg(std::max(1, c->smCount * 8 / gn), gn);
        nq::k_lab_bin_sum<<<bg, 256, 0, st>>>(gi, gs); ++c->launches;
      }
      nq::k_finalize_lab<<<n, 1024, 0, st>>>(dI, dS); ++c->launches;
      nq::k_lab_fewcolors<<<n, 256, 0, st>>>(dI, dS); ++c->launches;
    }
    mark(2);
    if (kind == NQ_KIND_RGB) {
      nq::k_rgb_blocks<<<dim3(2, n), 256, 0, st>>>(dI, dS); ++c->launches;
      nq::k_find_nn_all<<<c->smCount * 8, 256, 0, st>>>(dI, dS, n); ++c->launches;
    } else {
      nq::k_lab_blocks<<<dim3(2, n), 256, 0, st>>>(dI, dS); ++c->launches;
      nq::k_find_nn_lab<<<c->smCount * 8, 256, 0, st>>>(dI, dS, n); ++c->launches;
    }
    mark(3);
    if (c->debug) {
      CU(cudaStreamSynchronize(st));
      std::vector<NqImage> tmp(n);
      CU(cudaMemcpy(tmp.data(), dI, sizeof(NqImage) * n, cudaMemcpyDeviceToHost));
      for (int i = 0; i < n; ++i) {
        DebugImage& D = c->dbg[ch.base + i];
        const int mb = tmp[i].maxbins;
        const NqSlot& S = c->hSlots[ch.base + i];
        D.bins5.assign((size_t)mb * 5, 0.0);
        D.initErr.assign(mb, 0.f); D.initNn.assign(mb, 0);
        if (mb <= 0) continue;
        std::vector<double> col(mb);
        std::vector<float> colf(mb);
        for (int k = 0; k < 4; ++k) {
          if (kind == NQ_KIND_RGB) {
            const double* src = k == 0 ? S.bAc : k == 1 ? S.bC1 : k == 2 ? S.bC2 : S.bC3;
            CU(cudaMemcpy(col.data(), src, (size_t)mb * 8, cudaMemcpyDeviceToHost));
          } else {
            const float* src = k == 0 ? S.fAc : k == 1 ? S.fC1 : k == 2 ? S.fC2 : S.fC3;
            CU(cudaMemcpy(colf.data(), src, (size_t)mb * 4, cudaMemcpyDeviceToHost));
            for (int b = 0; b < mb; ++b) col[b] = colf[b];
          }
          for (int b = 0; b < mb; ++b) D.bins5[(size_t)b * 5 + k] = col[b];
        }
        CU(cudaMemcpy(colf.data(), S.bCnt, (size_t)mb * 4, cudaMemcpyDeviceToHost));
        for (int b = 0; b < mb; ++b) D.bins5[(size_t)b * 5 + 4] = colf[b];
        CU(cudaMemcpy(D.initErr.data(), S.bErr, (size_t)mb * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(D.initNn.data(), S.bNn, (size_t)mb * 4, cudaMemcpyDeviceToHost));
      }
    }
    if (A.stopAfterSweep) { mark(4); CU(cudaGetLastError()); return NQ_OK; }
    int* live = c->dLive + (size_t)ch.base * NQ_NBINS;
    int* pos = c->dPos + (size_t)ch.base * NQ_NBINS;
    if (kind == NQ_KIND_RGB) {
      nq::k_merge_rgb<<<n, NQ_RGB_THREADS, (size_t)NQ_RGB_HEAP_SMEM * 8, st>>>(dI, dS, live, pos, c->debug ? 1 : 0); ++c->launches;
    } else if (lab_merge_ctas(c, ch) == 8) {
      nq::k_merge_lab<8><<<n, NQ_LAB_THREADS, (size_t)nq::lab_heap_smem(8) * 8, st>>>(dI, dS, live, pos, c->debug ? 1 : 0); ++c->launches;
    } else {
      nq::k_merge_lab<4><<<n, NQ_LAB_THREADS, (size_t)nq::lab_heap_smem(4) * 8, st>>>(dI, dS, live, pos, c->debug ? 1 : 0); ++c->launches;
    }
  } else { mark(2); mark(3); }
  mark(4);
  CU(cudaGetLastError());
  return NQ_OK;
}

// dither of one chunk on the dither stream (after its front). The speculative path's rounds synchronise with the host;
// the serial kernels of the images it does not take run next to it on the aux stream.
int run_dither(nq_ctx* c, Chunk& ch, const GroupArgs& A, const uint32_t* dOrder) {
  NvtxRange nv("nq dither (setup, Gilbert pass, BlueNoise pass)");
  const int n = ch.n, npix = A.w * A.h, kind = A.kind;
  cudaStream_t st = c->sDith, ax = c->sAux;
  NqImage* dI = c->dImgs + ch.base;
  NqSlot* dS = c->dSlots + ch.base;
  unsigned long long l0 = c->launches;
  CU(cudaStreamWaitEvent(st, ch.ev[4], 0));
  CU(cudaEventRecord(ch.evD[0], st));
  nq::k_dither_setup<<<(n + 63) / 64, 64, 0, st>>>(dI, dS, n); ++c->launches;
  if (A.dPalIn) {
    for (int i = 0; i < n; ++i) { k_set_palette<<<1, 256, 0, st>>>(dI, i, A.dPalIn, A.palInLen); ++c->launches; }
    nq::k_dither_setup<<<(n + 63) / 64, 64, 0, st>>>(dI, dS, n); ++c->launches;
  }
  const dim3 pg(pixel_grid_x(c, npix, n), n);
  if (kind == NQ_KIND_LAB && c->debug) { nq::k_saliency<<<pg, 256, 0, st>>>(dI, dS); ++c->launches; }
  if (kind == NQ_KIND_LAB) { nq::k_build_cells<<<dim3(std::max(1, std::min(128, c->smCount * 8 / n)), n), 256, 0, st>>>(dI, dS); ++c->launches; }
  CU(cudaEventRecord(ch.evD[1], st));
  ch.launches[4] += c->launches - l0; l0 = c->launches;
  std::vector<int> elig, handed;
  const bool spec = c->specDither && kind == NQ_KIND_LAB && A.dither;
  SpecPlan plan;
  if (spec) {
    int rc = spec_prepare(c, ch, st, npix, dOrder, elig, &plan);
    if (rc) return rc;
  }
  // Everything the speculative path did not take (specDone == 0) goes through the serial kernels on the aux stream, next
  // to the speculative rounds; both kernels return at once for images of the other queue mode (decided on the device).
  const int cacheBytes = (kind == NQ_KIND_RGB || !A.dither) ? 32768 : 0;   // shared-memory memo cache when lookups stay on the chain
  cudaEvent_t evFork = take_event(c), evJoin = take_event(c);
  CU(cudaEventRecord(evFork, st));
  CU(cudaStreamWaitEvent(ax, evFork, 0));
  ch.evK[2] = take_event(c); ch.evK[3] = take_event(c);
  cudaEventRecord(ch.evK[2], ax);
  nq::k_dither_fifo<<<n, 64, cacheBytes, ax>>>(dI, dS, dOrder, cacheBytes, 0); ++c->launches;
  cudaEventRecord(ch.evK[3], ax);
  ch.evK[4] = take_event(c); ch.evK[5] = take_event(c);
  cudaEventRecord(ch.evK[4], ax);
  nq::k_dither_sorted<<<n, 32, 0, ax>>>(dI, dS, dOrder); ++c->launches;
  cudaEventRecord(ch.evK[5], ax);
  if (kind == NQ_KIND_RGB && !A.dither && A.nmax > 32) {   // BlueNoise.dither second pass, one thread per pixel (images flagged bnParallel)
    nq::k_bn_rgb_init<<<dim3(8, n), 256, 0, ax>>>(dI, dS); ++c->launches;
    nq::k_bn_rgb_a<<<pg, 256, 0, ax>>>(dI, dS); ++c->launches;
    nq::k_bn_rgb_b<<<dim3(16, n), 256, 0, ax>>>(dI, dS); ++c->launches;
    nq::k_bn_rgb_c<<<pg, 256, 0, ax>>>(dI, dS); ++c->launches;
  }
  if (spec) {
    int rc = spec_rounds(c, ch, st, npix, plan, elig, handed);
    if (rc) return rc;
    if (!handed.empty()) {   // qualifying images the rounds gave up on (specDone == 3): the serial kernel after all
      cudaEvent_t evBack = take_event(c);
      CU(cudaEventRecord(evBack, st));
      CU(cudaStreamWaitEvent(ax, evBack, 0));
      nq::k_dither_fifo<<<n, 64, cacheBytes, ax>>>(dI, dS, dOrder, cacheBytes, 3); ++c->launches;
    }
  }
  CU(cudaEventRecord(evJoin, ax));
  CU(cudaStreamWaitEvent(st, evJoin, 0));
  CU(cudaEventRecord(ch.evD[2], st));
  ch.launches[5] += c->launches - l0;
  CU(cudaGetLastError());
  return NQ_OK;
}

int check_args(nq_ctx* c, int kind, const void* in, int n, int w, int h, int nmax, const void* out) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  if (kind != NQ_KIND_PNN && kind != NQ_KIND_PNNLAB) return fail(NQ_ERR_ARG, "kind must be NQ_KIND_PNN or NQ_KIND_PNNLAB");
  if (!in || !out) return fail(NQ_ERR_ARG, "null pixel buffer");
  if (n <= 0 || w <= 0 || h <= 0) return fail(NQ_ERR_ARG, "n_images, width and height must be positive");
  if ((long long)w * h > 0x7fffffffLL / 4) return fail(NQ_ERR_ARG, "image too large");
  if (nmax < 2) return fail(NQ_ERR_ARG, "n_max_colors must be >= 2 (the reference indexes palette[1], PnnQuantizer.java:446)");
  if (nmax > NQ_MAXK) return fail(NQ_ERR_UNSUPPORTED, "n_max_colors > 256 is not supported by this build");
  return NQ_OK;
}

int collect_results(nq_ctx* c, int base, int n, uint32_t* palettes, int* plens, int* hasAlpha, int* firstErr) {
  for (int i = 0; i < n; ++i) {
    const NqImage& I = c->lastImgs[i];
    if (palettes) memcpy(palettes + (size_t)(base + i) * NQ_MAXK, I.palette, sizeof(uint32_t) * NQ_MAXK);
    if (plens) plens[base + i] = I.paletteLen;
    if (hasAlpha) hasAlpha[base + i] = I.transIdx > -1;
    if (I.error && !*firstErr) *firstErr = I.error;
  }
  return NQ_OK;
}

// convert() for images [0, n) of a group that fits the workspace: the group is cut into chunks that flow through
// front streams (scan .. merge), the dither stream and the copy-out stream, so that one chunk's merge loop, the previous
// chunk's dither and the host copies of both overlap. dIn / dOut are device buffers holding (or receiving, A.hIn) the pixels.
int convert_group(nq_ctx* c, const GroupArgs& A, int n, const uint32_t* dIn, uint32_t* dOut, int dbgBase) {
  const int npix = A.w * A.h;
  const uint32_t* dOrder = nullptr;
  int rc = ensure_order(c, A.w, A.h, &dOrder);
  if (rc) return rc;
  // Chunk sizes. The merge loop is the longest stage and its throughput grows with the images resident per SM, so a chunk
  // holds as many images as the merge kernel's resident CTAs on the whole device (k_merge_lab<8> for CIELAB: 1184 on 148
  // SMs, so a 1024-image batch runs all its merge loops in one wave, measured faster than two chunks of 512 on two front
  // streams). Host-buffer calls (from 32 images on) go in at least two, so that the copies of one piece overlap the kernels
  // of the other (a short first and last piece was tried and lost more in the merge loop than it hid). The device->host copy
  // of a chunk starts while its dither is still running (SpecCudaBackend::done_prefix).
  std::vector<int> sizes;
  if (c->debug) sizes.push_back(n);
  else if (c->chunkImages > 0) { for (int b = 0; b < n; b += c->chunkImages) sizes.push_back(std::min(c->chunkImages, n - b)); }
  else {
    const int slots = c->smCount * (A.kind == NQ_KIND_LAB ? c->mergeLab8PerSm : c->mergeRgbPerSm);
    const int pieces = std::max((n + slots - 1) / slots, (A.hIn && n >= 32) ? 2 : 1);
    for (int k = 0; k < pieces; ++k) sizes.push_back(n / pieces + (k < n % pieces ? 1 : 0));
  }
  const int nch = (int)sizes.size();
  c->evUsed = 0;
  std::vector<Chunk> chunks(nch);
  cudaEvent_t evStart = take_event(c), evOut = take_event(c), evEnd = take_event(c);
  CU(cudaEventRecord(evStart, c->stream));
  for (int k = 0; k < NQ_FRONT_STREAMS; ++k) CU(cudaStreamWaitEvent(c->sFront[k], evStart, 0));
  CU(cudaStreamWaitEvent(c->sDith, evStart, 0));
  CU(cudaStreamWaitEvent(c->sOut, evStart, 0));
  CU(cudaStreamWaitEvent(c->sIn, evStart, 0));
  for (int k = 0, base = 0; k < nch; base += sizes[k], ++k) {
    Chunk& ch = chunks[k];
    ch.base = base; ch.n = sizes[k];
    ch.mergeInFlight = sizes[k] + std::max(k > 0 ? sizes[k - 1] : 0, k + 1 < nch ? sizes[k + 1] : 0);   // two front streams
    ch.frontIdx = k % NQ_FRONT_STREAMS; ch.front = c->sFront[ch.frontIdx];
    for (auto& e : ch.ev) e = take_event(c);
    for (auto& e : ch.evD) e = take_event(c);
    if (A.hIn) {   // every chunk's pixels are copied in on their own stream, in order, as early as the copy engine allows
      ch.evIn = take_event(c);
      CU(cudaMemcpyAsync(const_cast<uint32_t*>(dIn) + (size_t)ch.base * npix, A.hIn + (size_t)ch.base * npix, (size_t)ch.n * npix * 4, cudaMemcpyHostToDevice, c->sIn));
      CU(cudaEventRecord(ch.evIn, c->sIn));
    }
  }
  if (c->debug) for (int i = 0; i < n; ++i) c->dbg[dbgBase + i] = DebugImage{};
  GroupArgs G = A;
  // every front is enqueued before the first dither (the speculative rounds block this thread); consecutive chunks
  // alternate between the front streams, so at most two merge loops run next to each other and next to a dither
  for (int k = 0; k < nch; ++k) { rc = enqueue_front(c, chunks[k], G, dIn, dOut); if (rc) return rc; }
  for (int k = 0; k < nch; ++k) {
    if (A.stopAfterSweep) {   // the dither stream only has to wait for the front
      CU(cudaStreamWaitEvent(c->sDith, chunks[k].ev[4], 0));
      for (auto& e : chunks[k].evD) CU(cudaEventRecord(e, c->sDith));
      continue;
    }
    if (A.hOut) { chunks[k].hOut = A.hOut + (size_t)chunks[k].base * npix; chunks[k].dOut = dOut + (size_t)chunks[k].base * npix; chunks[k].imageBytes = (size_t)npix * 4; }
    rc = run_dither(c, chunks[k], G, dOrder);
    if (rc) return rc;
    if (A.hOut && chunks[k].copied < chunks[k].n) {   // device -> host of what the progressive copy-out has not taken yet
      Chunk& ch = chunks[k];
      CU(cudaStreamWaitEvent(c->sOut, ch.evD[2], 0));
      CU(cudaMemcpyAsync(A.hOut + (size_t)(ch.base + ch.copied) * npix, dOut + (size_t)(ch.base + ch.copied) * npix, (size_t)(ch.n - ch.copied) * npix * 4,
                         cudaMemcpyDeviceToHost, c->sOut));
    }
  }
  CU(cudaEventRecord(evOut, c->sOut));
  CU(cudaStreamWaitEvent(c->sDith, evOut, 0));
  c->lastImgs.resize(n);
  CU(cudaMemcpyAsync(c->lastImgs.data(), c->dImgs, sizeof(NqImage) * n, cudaMemcpyDeviceToHost, c->sDith));
  CU(cudaEventRecord(evEnd, c->sDith));
  CU(cudaStreamWaitEvent(c->stream, evEnd, 0));     // the caller's stream is ordered behind the whole call
  CU(cudaStreamSynchronize(c->sDith));
  for (int k = 0; k < NQ_FRONT_STREAMS; ++k) CU(cudaStreamSynchronize(c->sFront[k]));
  CU(cudaStreamSynchronize(c->sAux));
  CU(cudaStreamSynchronize(c->sIn));
  for (Chunk& ch : chunks) {
    float ms = 0.f;
    for (int k = 0; k < 4; ++k) if (cudaEventElapsedTime(&ms, ch.ev[k], ch.ev[k + 1]) == cudaSuccess) c->stageMs[k] += ms;
    for (int k = 0; k < 2; ++k) if (cudaEventElapsedTime(&ms, ch.evD[k], ch.evD[k + 1]) == cudaSuccess) c->stageMs[4 + k] += ms;
    for (int k = 0; k < NQ_NSTAGES; ++k) c->stageLaunches[k] += ch.launches[k];
    for (auto& pr : ch.evRuns) if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) { c->kernelMs[0] += ms; ++c->kernelLaunches[0]; }
    for (int k = 1; k < NQ_NKERNELS; ++k)
      if (ch.evK[2 * k] && cudaEventElapsedTime(&ms, ch.evK[2 * k], ch.evK[2 * k + 1]) == cudaSuccess) { c->kernelMs[k] += ms; ++c->kernelLaunches[k]; }
    if (cudaEventElapsedTime(&ms, ch.ev[3], ch.ev[4]) == cudaSuccess) { c->kernelMs[3] += ms; ++c->kernelLaunches[3]; }
  }
  cudaGetLastError();
  if (getenv("NQ_SPEC_TIMING") || getenv("NQ_SPEC_REASONS"))
    for (int i = 0; i < n; ++i)
      if (c->lastImgs[i].specDone == 3) fprintf(stderr, "[nq spec] image %d handed back to the serial kernel, reason %d\n", i, c->lastImgs[i].pad1);
  if (c->debug) {
    for (int i = 0; i < n; ++i) {
      DebugImage& D = c->dbg[dbgBase + i];
      const NqImage& I = c->lastImgs[i];
      const int merges = (A.nmax > 2 && I.extbins > 0) ? I.extbins : 0;
      D.merges.assign((size_t)merges * 2, 0);
      if (merges && c->hSlots[i].mergeLog) CU(cudaMemcpy(D.merges.data(), c->hSlots[i].mergeLog, (size_t)merges * 8, cudaMemcpyDeviceToHost));
      D.sal.clear();
      if (I.gUseSal && c->hSlots[i].sal) { D.sal.resize(npix); CU(cudaMemcpy(D.sal.data(), c->hSlots[i].sal, (size_t)npix * 4, cudaMemcpyDeviceToHost)); }
    }
  }
  return NQ_OK;
}

// dIn / dOut: device buffers for the whole batch. hIn / hOut (optional): host buffers the batch is read from / written to
// chunk by chunk, overlapped with the kernels.
int convert_device(nq_ctx* c, int kind, const uint32_t* dIn, int n, int w, int h, int nmax, int dither, const uint64_t* seeds,
                   uint32_t* dOut, uint32_t* palettes, int* plens, int* hasAlpha, const uint32_t* dPalIn, int palInLen,
                   const uint32_t* hIn = nullptr, uint32_t* hOut = nullptr, bool stopAfterSweep = false) {
  CU(cudaSetDevice(c->device));
  const int npix = w * h;
  // the BlueNoise second pass of PnnLABQuantizer weighs by pixelMap.size() (PL:511-513): track it only then
  const bool needBits = kind == NQ_KIND_LAB && !dither && nmax > 32;
  // PnnQuantizer's BlueNoise second pass runs one thread per pixel and keeps the first-pass indices next to the output
  const bool needIdx = kind == NQ_KIND_RGB && !dither && nmax > 32;
  int rc = ensure_workspace(c, kind, npix, n, needBits, needIdx);
  if (rc) return rc;
  if (c->debug) c->dbg.assign(n, DebugImage{});
  int firstErr = 0;
  std::vector<NqImage> all;
  all.reserve(n);
  for (int base = 0; base < n; base += c->wsSlots) {
    const int m = std::min(c->wsSlots, n - base);
    GroupArgs A{kind, w, h, nmax, dither, seeds ? seeds + base : nullptr, dPalIn, palInLen,
                hIn ? hIn + (size_t)base * npix : nullptr, hOut ? hOut + (size_t)base * npix : nullptr};
    A.stopAfterSweep = stopAfterSweep;
    rc = convert_group(c, A, m, dIn + (size_t)base * npix, dOut + (size_t)base * npix, base);
    if (rc) return rc;
    collect_results(c, base, m, palettes, plens, hasAlpha, &firstErr);
    all.insert(all.end(), c->lastImgs.begin(), c->lastImgs.end());
  }
  c->lastImgs.swap(all);
  if (firstErr == 3) return fail(NQ_ERR_COLOR, "alpha must be between 0 and 255. (ColorUtils.setAlphaComponent)");
  if (firstErr == 4) return fail(NQ_ERR_UNSUPPORTED, "PnnLABQuantizer with dither == false, more than 32 colours and semi-transparent pixels is not covered");
  if (firstErr) return fail(NQ_ERR_UNSUPPORTED, "device-side error " + std::to_string(firstErr));
  return NQ_OK;
}

int ensure_stage(nq_ctx* c, size_t bytes) {
  if (c->stageBytes >= bytes) return NQ_OK;
  CU(cudaDeviceSynchronize());
  if (c->dIn) cudaFree(c->dIn);
  if (c->dOut) cudaFree(c->dOut);
  c->dIn = c->dOut = nullptr; c->stageBytes = 0;
  CU(cudaMalloc(&c->dIn, bytes));
  cudaError_t e = cudaMalloc(&c->dOut, bytes);
  if (e != cudaSuccess) { cudaFree(c->dIn); c->dIn = nullptr; return fail(NQ_ERR_NOMEM, std::string("cudaMalloc(staging): ") + cudaGetErrorString(e)); }
  c->stageBytes = bytes;
  return NQ_OK;
}

}  // namespace

namespace {
void destroy_ctx(nq_ctx* c, bool dropLut) {
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (dropLut) {
    std::lock_guard<std::mutex> lk(g_lutMutex);
    auto it = g_lut.find(c->device);
    if (it != g_lut.end() && it->second.refs > 0 && --it->second.refs == 0) { cudaFree(it->second.ptr); g_lut.erase(it); }
  }
  for (auto& kv : c->orders) cudaFree(kv.second);
  if (c->ws) cudaFree(c->ws);
  if (c->dIn) cudaFree(c->dIn);
  if (c->dOut) cudaFree(c->dOut);
  if (c->dSpec) cudaFree(c->dSpec);
  if (c->specBuf) cudaFree(c->specBuf);
  if (c->dSpecPool) cudaFree(c->dSpecPool);
  if (c->dSpecInts) cudaFree(c->dSpecInts);
  if (c->dTanh) cudaFree(c->dTanh);
  for (cudaEvent_t e : c->evPool) if (e) cudaEventDestroy(e);
  for (int k = 0; k < NQ_FRONT_STREAMS; ++k) if (c->sFront[k]) cudaStreamDestroy(c->sFront[k]);
  if (c->sDith) cudaStreamDestroy(c->sDith);
  if (c->sAux) cudaStreamDestroy(c->sAux);
  if (c->sOut) cudaStreamDestroy(c->sOut);
  if (c->sIn) cudaStreamDestroy(c->sIn);
  if (c->ownStream) cudaStreamDestroy(c->ownStream);
  delete c;
}
// temporary device buffers of the probe / hook entry points: freed on every exit
struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes); }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};
__global__ void k_spec_tables(float* tanhTab, float* w3) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < 511) tanhTab[t] = nq::spec::tanh_f((double)((float)(t - 255) / 255.f * 20.f));
  if (t < 3) {   // initWeights(9 | 16 | 25), padded to NQ_MAXQ + 3 floats per row (GC:336-354)
    const int DM = t == 0 ? 9 : (t == 1 ? 16 : 25);
    float w[NQ_MAXQ];
    nq::init_weights(w, DM);
    for (int k = 0; k < NQ_MAXQ + 3; ++k) w3[t * (NQ_MAXQ + 3) + k] = k < DM ? w[k] : 0.f;
  }
}
}  // namespace

extern "C" {

int nq_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

const char* nq_last_error(void) { return g_lastError.c_str(); }

nq_ctx* nq_create(int device) {
  int n = nq_device_count();
  if (device < 0 || device >= n) { fail(NQ_ERR_CUDA, "no such CUDA device (this library has no CPU fallback)"); return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { fail(NQ_ERR_CUDA, "cudaSetDevice failed"); return nullptr; }
  nq_ctx* c = new nq_ctx();
  c->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->smCount = prop.multiProcessorCount;
  bool ok = cudaStreamCreateWithFlags(&c->ownStream, cudaStreamNonBlocking) == cudaSuccess;
  for (int k = 0; ok && k < NQ_FRONT_STREAMS; ++k) ok = cudaStreamCreateWithFlags(&c->sFront[k], cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&c->sDith, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&c->sAux, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&c->sOut, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&c->sIn, cudaStreamNonBlocking) == cudaSuccess;
  if (!ok) { fail(NQ_ERR_CUDA, "cudaStreamCreate failed"); destroy_ctx(c, false); return nullptr; }
  c->stream = c->ownStream;
  if (const char* e = getenv("NQ_SPEC_DITHER")) c->specDither = atoi(e) != 0;
  if (const char* e = getenv("NQ_CHUNK")) c->chunkImages = atoi(e);
  {
    const char* e = getenv("NQ_SPEC_BULK");
    const int bulk = e ? (atoi(e) != 0) : NQ_SPEC_BULK_DEFAULT;
    ok = ok && cudaMemcpyToSymbol(nq::spec::g_specBulk, &bulk, sizeof(bulk)) == cudaSuccess;
  }
  if (const char* e = getenv("NQ_SPEC_SLOTS")) c->specSlotsMax = atoi(e);
  if (const char* e = getenv("NQ_SPEC_POOL_GB")) c->specPoolMaxBytes = (size_t)atoi(e) << 30;
  bool haveLut = false;
  {
    DevBuf dBn, dW;
    ok = dBn.alloc(4096) == cudaSuccess && cudaMemcpy(dBn.p, kBlueNoise, 4096, cudaMemcpyHostToDevice) == cudaSuccess &&
         dW.alloc(sizeof(float) * 3 * (NQ_MAXQ + 3)) == cudaSuccess && cudaMalloc(&c->dTanh, sizeof(float) * 512) == cudaSuccess;
    if (ok) {
      nq::k_init_tables<<<4, 256, 0, c->stream>>>(dBn.as<signed char>()); ++c->launches;
      nq::k_init_rtfac<<<1, 256, 0, c->stream>>>(); ++c->launches;
      k_spec_tables<<<2, 256, 0, c->stream>>>(c->dTanh, dW.as<float>()); ++c->launches;
      ok = cudaMemcpyToSymbolAsync(nq::spec::c_specW, dW.p, sizeof(float) * 3 * (NQ_MAXQ + 3), 0, cudaMemcpyDeviceToDevice, c->stream) == cudaSuccess &&
           cudaStreamSynchronize(c->stream) == cudaSuccess;
    }
  }
  if (ok) {
    std::lock_guard<std::mutex> lk(g_lutMutex);
    LabLutEntry& e = g_lut[device];
    if (!e.ptr) {
      ok = cudaMalloc(&e.ptr, sizeof(float4) << 24) == cudaSuccess;
      if (ok) {
        nq::k_build_lab_lut<<<65536, 256, 0, c->stream>>>(e.ptr); ++c->launches;
        const float4* cp = e.ptr;
        ok = cudaMemcpyToSymbolAsync(nq::g_labLut, &cp, sizeof(cp), 0, cudaMemcpyHostToDevice, c->stream) == cudaSuccess &&
             cudaStreamSynchronize(c->stream) == cudaSuccess;
      }
      if (!ok && e.ptr) { cudaFree(e.ptr); e.ptr = nullptr; }
    }
    if (ok) { ++e.refs; haveLut = true; }
  }
  if (ok) ok = cudaFuncSetAttribute(nq::k_merge_rgb, cudaFuncAttributeMaxDynamicSharedMemorySize, NQ_RGB_HEAP_SMEM * 8) == cudaSuccess;
  if (ok) ok = cudaFuncSetAttribute(nq::k_hist_rgb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(nq::HistTable)) == cudaSuccess;
  if (ok) ok = cudaFuncSetAttribute(nq::k_dither_fifo, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768) == cudaSuccess;
  if (ok) ok = cudaFuncSetAttribute(nq::k_merge_lab<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, nq::lab_heap_smem(4) * 8) == cudaSuccess &&
               cudaFuncSetAttribute(nq::k_merge_lab<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, nq::lab_heap_smem(8) * 8) == cudaSuccess;
  if (ok) ok = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->mergeLab4PerSm, nq::k_merge_lab<4>, NQ_LAB_THREADS, nq::lab_heap_smem(4) * 8) == cudaSuccess &&
               cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->mergeLab8PerSm, nq::k_merge_lab<8>, NQ_LAB_THREADS, nq::lab_heap_smem(8) * 8) == cudaSuccess &&
               cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c->mergeRgbPerSm, nq::k_merge_rgb, NQ_RGB_THREADS, NQ_RGB_HEAP_SMEM * 8) == cudaSuccess &&
               c->mergeLab4PerSm > 0 && c->mergeLab8PerSm > 0 && c->mergeRgbPerSm > 0;
  if (!ok) {
    fail(NQ_ERR_CUDA, std::string("context initialisation failed: ") + cudaGetErrorString(cudaGetLastError()));
    destroy_ctx(c, haveLut);          // drops the table reference taken above, the streams and every allocation
    return nullptr;
  }
  return c;
}

void nq_destroy(nq_ctx* c) {
  if (!c) return;
  destroy_ctx(c, true);
}

int nq_convert_batch_device(nq_ctx* c, int kind, const uint32_t* d_in, int n, int w, int h, int nmax, int dither,
                            const uint64_t* seeds, uint32_t* d_out, uint32_t* palettes, int* plens, int* hasAlpha) {
  int rc = check_args(c, kind, d_in, n, w, h, nmax, d_out);
  if (rc) return rc;
  NvtxRange nv("nq_convert_batch_device");
  return convert_device(c, kind, d_in, n, w, h, nmax, dither, seeds, d_out, palettes, plens, hasAlpha, nullptr, 0);
}

int nq_convert_batch(nq_ctx* c, int kind, const uint32_t* in, int n, int w, int h, int nmax, int dither, const uint64_t* seeds,
                     uint32_t* out, uint32_t* palettes, int* plens, int* hasAlpha) {
  int rc = check_args(c, kind, in, n, w, h, nmax, out);
  if (rc) return rc;
  NvtxRange nv("nq_convert_batch");
  CU(cudaSetDevice(c->device));
  const size_t bytes = (size_t)n * w * h * 4;
  rc = ensure_stage(c, bytes);
  if (rc) return rc;
  // host -> device, kernels and device -> host are interleaved chunk by chunk inside convert_device
  rc = convert_device(c, kind, c->dIn, n, w, h, nmax, dither, seeds, c->dOut, palettes, plens, hasAlpha, nullptr, 0, in, out);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream));
  return NQ_OK;
}

// One worker thread per context pulls pieces of the batch from a shared counter (a dynamic queue: a GPU that finishes early
// takes the next piece) and runs nq_convert_batch on its piece. No collective: the images are independent.
int nq_convert_batch_multi(nq_ctx** ctxs, int nctx, int kind, const uint32_t* in, int n, int w, int h, int nmax, int dither,
                           const uint64_t* seeds, uint32_t* out, uint32_t* palettes, int* plens, int* hasAlpha, int queueImages) {
  if (!ctxs || nctx <= 0) return fail(NQ_ERR_ARG, "no contexts");
  for (int g = 0; g < nctx; ++g) if (!ctxs[g]) return fail(NQ_ERR_ARG, "null context in the list");
  int rc = check_args(ctxs[0], kind, in, n, w, h, nmax, out);
  if (rc) return rc;
  if (queueImages < 0) return fail(NQ_ERR_ARG, "queue_images must be >= 0");
  const int piece = queueImages > 0 ? queueImages : (n + nctx - 1) / nctx;   // default: one piece per context
  const size_t npix = (size_t)w * h;
  std::atomic<int> next(0), firstRc(NQ_OK);
  std::mutex errMutex;
  std::string errMsg;
  auto worker = [&](int g) {
    for (;;) {
      const int base = next.fetch_add(piece);
      if (base >= n || firstRc.load() != NQ_OK) return;
      const int m = std::min(piece, n - base);
      const int r = nq_convert_batch(ctxs[g], kind, in + (size_t)base * npix, m, w, h, nmax, dither, seeds ? seeds + base : nullptr,
                                     out + (size_t)base * npix, palettes ? palettes + (size_t)base * NQ_MAXK : nullptr,
                                     plens ? plens + base : nullptr, hasAlpha ? hasAlpha + base : nullptr);
      if (r != NQ_OK) {
        std::lock_guard<std::mutex> lk(errMutex);
        int expected = NQ_OK;
        if (firstRc.compare_exchange_strong(expected, r)) errMsg = "context " + std::to_string(g) + ", images " + std::to_string(base) + ".." + std::to_string(base + m - 1) + ": " + nq_last_error();
        return;
      }
    }
  };
  std::vector<std::thread> threads;
  for (int g = 1; g < nctx; ++g) threads.emplace_back(worker, g);
  worker(0);
  for (auto& t : threads) t.join();
  if (firstRc.load() != NQ_OK) return fail(firstRc.load(), errMsg);
  return NQ_OK;
}

int nq_convert(nq_ctx* c, int kind, const uint32_t* in, int w, int h, int nmax, int dither, uint64_t seed, uint32_t* out,
               uint32_t* palette, int* plen, int* hasAlpha) {
  return nq_convert_batch(c, kind, in, 1, w, h, nmax, dither, &seed, out, palette, plen, hasAlpha);
}

int nq_dither_with_palette(nq_ctx* c, int kind, const uint32_t* in, int w, int h, int nmax, int dither, uint64_t seed,
                           const uint32_t* palette, int plen, uint32_t* out) {
  int rc = check_args(c, kind, in, 1, w, h, nmax, out);
  if (rc) return rc;
  if (!palette || plen <= 0 || plen > NQ_MAXK) return fail(NQ_ERR_ARG, "palette_len must be 1..256");
  CU(cudaSetDevice(c->device));
  const size_t bytes = (size_t)w * h * 4;
  rc = ensure_stage(c, bytes);
  if (rc) return rc;
  DevBuf dPal;
  CU(dPal.alloc(NQ_MAXK * 4));
  CU(cudaMemcpy(dPal.p, palette, (size_t)plen * 4, cudaMemcpyHostToDevice));
  rc = convert_device(c, kind, c->dIn, 1, w, h, nmax, dither, &seed, c->dOut, nullptr, nullptr, nullptr, dPal.as<uint32_t>(), plen, in, out);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream));
  return NQ_OK;
}

int nq_histogram(nq_ctx* c, int kind, const uint32_t* in, int w, int h, int nmax, int* nBins, double* bins5, float* initErr, int* initNn, int capacity) {
  int rc = check_args(c, kind, in, 1, w, h, nmax, in);
  if (rc) return rc;
  if (!nBins) return fail(NQ_ERR_ARG, "n_bins must not be null");
  CU(cudaSetDevice(c->device));
  const size_t bytes = (size_t)w * h * 4;
  rc = ensure_stage(c, bytes);
  if (rc) return rc;
  const bool wasDebug = c->debug;
  c->debug = true;                                   // the hook returns what debug mode records after the find_nn sweep
  uint64_t seed = 0;
  rc = convert_device(c, kind, c->dIn, 1, w, h, nmax, 1, &seed, c->dOut, nullptr, nullptr, nullptr, nullptr, 0, in, nullptr, true);
  c->debug = wasDebug;
  if (rc) return rc;
  const DebugImage& D = c->dbg[0];
  const int mb = (int)D.initErr.size();
  *nBins = mb;
  if (mb > capacity && (bins5 || initErr || initNn)) return fail(NQ_ERR_ARG, "capacity is smaller than the number of occupied bins (call with null outputs to size them)");
  if (bins5) memcpy(bins5, D.bins5.data(), D.bins5.size() * 8);
  if (initErr) memcpy(initErr, D.initErr.data(), D.initErr.size() * 4);
  if (initNn) memcpy(initNn, D.initNn.data(), D.initNn.size() * 4);
  return NQ_OK;
}

int nq_gilbert_order(int w, int h, uint32_t* out) {
  if (w <= 0 || h <= 0 || !out) return fail(NQ_ERR_ARG, "bad arguments");
  size_t n = 0;
  gilbert_walk(w, h, [&](int x, int y) { out[n++] = (uint32_t)(x + y * w); });
  return n == (size_t)w * h ? NQ_OK : fail(NQ_ERR_ARG, "gilbert walk size mismatch");
}

int nq_get_image_info(nq_ctx* c, int image, nq_image_info* o) {
  if (!c || !o || image < 0 || image >= (int)c->lastImgs.size()) return fail(NQ_ERR_ARG, "no such image in the last batch");
  const NqImage& I = c->lastImgs[image];
  memset(o, 0, sizeof(*o));
  o->has_semi_transparency = I.hasSemi; o->transparent_pixel_index = I.transIdx; o->transparent_color = I.transColor;
  o->maxbins = I.maxbins; o->quan_rt = I.quan_rt; o->texicab = I.texicab; o->is_nano = I.isNano;
  o->weight = I.weight; o->ratio_init = I.ratio; o->ratio_merge = I.ratioMerge;
  o->pr = I.PR; o->pg = I.PG; o->pb = I.PB; o->pa = I.PA;
  o->g_margin = I.gMargin; o->g_thresold = I.gThresold; o->g_dither_max_q = I.gDitherMaxQ; o->g_dither_max = I.gDitherMax;
  o->g_sorted = I.gSorted; o->g_has_alpha = I.gHasAlpha; o->g_use_saliency = I.gUseSal; o->g_beta = I.gBeta;
  o->bn_weight = I.bnWeight; o->palette_len = I.paletteLen;
  o->merges = (I.nmax > 2 && I.extbins > 0) ? (unsigned long long)I.extbins : 0ULL;
  o->rescans = I.statRescans; o->pair_tests = I.statPairs; o->rng_draws = I.rngDraws; o->heap_pops = I.statHeapPops;
  o->full_evals = I.statFullEvals;
  for (int k = 0; k < 6; ++k) o->merge_cycles[k] = I.statCyc[k];
  o->live_blocks = I.statLiveBlocks; o->screened = I.statScreened;
  o->merge_rounds = I.statRounds; o->rescans_discarded = I.statDiscarded;
  o->merge_ctas_per_sm = I.mergeCtas;
  for (int k = 0; k < 3; ++k) o->dither_cycles[k] = I.statDither[k];
  o->error = I.error;
  return NQ_OK;
}

int nq_sizeof_image_info(void) { return (int)sizeof(nq_image_info); }

int nq_set_stream(nq_ctx* c, void* stream) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  // a NULL handle is CUDA's legacy default stream (what torch.cuda.default_stream().cuda_stream is), not "our own"
  c->stream = stream ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamLegacy;
  return NQ_OK;
}
int nq_reset_stream(nq_ctx* c) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  c->stream = c->ownStream;
  return NQ_OK;
}
int nq_set_chunk_images(nq_ctx* c, int images) {
  if (!c || images < 0) return fail(NQ_ERR_ARG, "bad arguments");
  c->chunkImages = images;
  return NQ_OK;
}

int nq_set_spec_dither(nq_ctx* c, int on, int segment, int warmup) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  if (on && ((segment != 0 && segment < 64) || warmup < 0 || warmup > (1 << 24))) return fail(NQ_ERR_ARG, "segment must be 0 (automatic) or >= 64 pixels, warm-up >= 0");
  c->specDither = on != 0;
  if (on) { c->specSeg = segment; c->specWarm = warmup; }
  return NQ_OK;
}
int nq_get_spec_stats(nq_ctx* c, unsigned long long* images, unsigned long long* rounds, unsigned long long* fallbacks) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  if (images) *images = c->specImages;
  if (rounds) *rounds = c->specRounds;
  if (fallbacks) *fallbacks = c->specFallbacks;
  return NQ_OK;
}

int nq_set_debug(nq_ctx* c, int flag) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  c->debug = flag != 0;
  return NQ_OK;
}

int nq_debug_get_bins(nq_ctx* c, int image, double* bins5, float* initErr, int* initNn) {
  if (!c || image < 0 || image >= (int)c->dbg.size()) return fail(NQ_ERR_ARG, "no debug record for that image");
  const DebugImage& D = c->dbg[image];
  if (bins5) memcpy(bins5, D.bins5.data(), D.bins5.size() * 8);
  if (initErr) memcpy(initErr, D.initErr.data(), D.initErr.size() * 4);
  if (initNn) memcpy(initNn, D.initNn.data(), D.initNn.size() * 4);
  return NQ_OK;
}
int nq_debug_get_merges(nq_ctx* c, int image, int* pairs) {
  if (!c || image < 0 || image >= (int)c->dbg.size()) return fail(NQ_ERR_ARG, "no debug record for that image");
  const DebugImage& D = c->dbg[image];
  if (pairs) memcpy(pairs, D.merges.data(), D.merges.size() * 4);
  return NQ_OK;
}
int nq_debug_get_saliencies(nq_ctx* c, int image, float* out) {
  if (!c || image < 0 || image >= (int)c->dbg.size()) return fail(NQ_ERR_ARG, "no debug record for that image");
  const DebugImage& D = c->dbg[image];
  if (D.sal.empty()) return fail(NQ_ERR_ARG, "this image has no saliency map");
  if (out) memcpy(out, D.sal.data(), D.sal.size() * 4);
  return NQ_OK;
}

unsigned long long nq_kernel_launches(nq_ctx* c) { return c ? c->launches : 0ULL; }

int nq_get_stage_times(nq_ctx* c, double* ms, unsigned long long* launches, int reset) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  for (int k = 0; k < NQ_NSTAGES; ++k) {
    if (ms) ms[k] = c->stageMs[k];
    if (launches) launches[k] = c->stageLaunches[k];
    if (reset) { c->stageMs[k] = 0; c->stageLaunches[k] = 0; }
  }
  return NQ_OK;
}
int nq_get_kernel_times(nq_ctx* c, double* ms, unsigned long long* launches, int reset) {
  if (!c) return fail(NQ_ERR_ARG, "null context");
  for (int k = 0; k < NQ_NKERNELS; ++k) {
    if (ms) ms[k] = c->kernelMs[k];
    if (launches) launches[k] = c->kernelLaunches[k];
    if (reset) { c->kernelMs[k] = 0; c->kernelLaunches[k] = 0; }
  }
  return NQ_OK;
}

int nq_debug_math(nq_ctx* c, int fn, const double* x, const double* y, double* out, int n) {
  if (!c || !x || !out || n <= 0) return fail(NQ_ERR_ARG, "bad arguments");
  CU(cudaSetDevice(c->device));
  DevBuf dx, dy, dout;
  CU(dx.alloc((size_t)n * 8));
  CU(dy.alloc((size_t)n * 8));
  CU(dout.alloc((size_t)n * 8));
  CU(cudaMemcpy(dx.p, x, (size_t)n * 8, cudaMemcpyHostToDevice));
  if (y) CU(cudaMemcpy(dy.p, y, (size_t)n * 8, cudaMemcpyHostToDevice));
  else CU(cudaMemset(dy.p, 0, (size_t)n * 8));
  k_math_probe<<<(n + 127) / 128, 128, 0, c->ownStream>>>(fn, dx.as<double>(), dy.as<double>(), dout.as<double>(), n); ++c->launches;
  CU(cudaStreamSynchronize(c->ownStream));
  CU(cudaMemcpy(out, dout.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
  return NQ_OK;
}

int nq_debug_ciede(nq_ctx* c, const float* lab1, const float* lab2, float* out, int* nExact, int n) {
  if (!c || !lab1 || !lab2 || !out || n <= 0) return fail(NQ_ERR_ARG, "bad arguments");
  CU(cudaSetDevice(c->device));
  DevBuf d1, d2, dout, dcnt;
  CU(d1.alloc((size_t)n * 12));
  CU(d2.alloc((size_t)n * 12));
  CU(dout.alloc((size_t)n * 16));
  CU(dcnt.alloc(4));
  CU(cudaMemcpy(d1.p, lab1, (size_t)n * 12, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d2.p, lab2, (size_t)n * 12, cudaMemcpyHostToDevice));
  CU(cudaMemset(dcnt.p, 0, 4));
  k_ciede_probe<<<(n + 127) / 128, 128, 0, c->ownStream>>>(d1.as<float>(), d2.as<float>(), dout.as<float>(), dcnt.as<int>(), n); ++c->launches;
  CU(cudaStreamSynchronize(c->ownStream));
  CU(cudaMemcpy(out, dout.p, (size_t)n * 16, cudaMemcpyDeviceToHost));
  int cnt = 0;
  CU(cudaMemcpy(&cnt, dcnt.p, 4, cudaMemcpyDeviceToHost));
  if (nExact) *nExact = cnt;
  return NQ_OK;
}

int nq_synth_device(nq_ctx* c, uint32_t* d_out, int n, int w, int h, int cls, int amode, uint64_t seed0) {
  if (!c || !d_out || n <= 0 || w <= 0 || h <= 0) return fail(NQ_ERR_ARG, "bad arguments");
  CU(cudaSetDevice(c->device));
  k_synth<<<c->smCount * 8, 256, 0, c->stream>>>(d_out, n, w, h, cls, amode, seed0); ++c->launches;
  CU(cudaStreamSynchronize(c->stream));
  return NQ_OK;
}

}  // extern "C"
