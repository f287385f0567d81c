// nq_types.h -- per-image device record and workspace layout shared by all stage kernels.
#pragma once
#include <stdint.h>

#define NQ_MAXK 256          // largest palette the CUDA path handles (BASELINE.json sweeps 2..256)
#define NQ_NBINS 65536       // histogram bins (PQ:137, PL:134)
#define NQ_DELETED 0xFFFF    // mtm marker of a merged-away bin (PQ:220,254)
#define NQ_MAXQ 25           // largest DITHER_MAX (GC:96)

enum NqKind { NQ_KIND_RGB = 0, NQ_KIND_LAB = 1 };

// Everything convert() derives per image lives here, in device memory, so a whole batch runs
// stage after stage without a host round trip.
struct NqImage {
  // inputs
  int kind, width, height, npix, nmax, dither;
  unsigned long long seed;
  // alpha scan (PQ:411-431)
  unsigned int semiCount;
  int transIdx;            // m_transparentPixelIndex
  int hasSemi;             // hasSemiTransparency
  uint32_t transColor;     // m_transparentColor
  int fixA0;               // nMaxColors <= 2: a==0 pixels are rewritten to 0x00FFFFFF (PQ:424)
  int keyTransp;           // 3rd argument of getColorIndex in pnnquan (PQ:144)
  // pnnquan scalars
  int maxbins, extbins, quan_rt, texicab, isNano, skipPnn;
  double PR, PG, PB, PA, ratio, ratioMerge, weight;
  // palette
  int paletteLen;
  uint32_t palette[NQ_MAXK];
  // GilbertCurve constructor (GC:50-112)
  int gMargin, gThresold, gDitherMaxQ /*DITHER_MAX*/, gDitherMax, gSorted, gHasAlpha, gUseSal;
  float gBeta;
  double gWeight;          // |weight|
  float gWeights[NQ_MAXQ]; // initWeights(DITHER_MAX) for the FIFO queue
  float gW1[1], gW3[3], gW7[7];  // initWeights(1|3|7) for the sorted queue warm-up (GC:233-234)
  float bnWeight;          // weight of the BlueNoise second pass
  int error;               // 0 ok, else NQ_ERR_* raised on the device
  // statistics
  unsigned long long statRescans, statPairs, rngDraws, statFullEvals;
  unsigned int statHeapPops;
  unsigned int distinctColors;     // pixelMap.size() so far (only tracked when NqSlot::bits is set)
  // merge-loop phase clocks (SM cycles, thread 0): 0 heap/top, 1 first-32, 2 block tests, 3 screen, 4 full+resolve, 5 merge+rebuild
  unsigned long long statCyc[6], statLiveBlocks, statScreened;
  unsigned long long statRounds, statDiscarded;   // CIELAB merge loop: rescan rounds, rescans computed but not applied
  int mergeCtas;                                  // resident CTAs per SM of the merge loop instance launched (set by the host)
  unsigned long long statDither[3];   // FIFO dither: consumer cycles, consumer cycles waiting for the producer, producer cycles waiting
  int specDone;            // speculative segment-parallel dither (nq_dither_spec.cuh): 0 not its image, 1 dithered by it, 2 pending there,
                           // 3 handed back to k_dither_fifo
  unsigned int nonOpaque;  // pixels whose alpha is not 255 (alpha scan)
  int bnParallel;          // BlueNoise.dither second pass done by the per-pixel kernels k_bn_* instead of the serial warp
  int pad1;
};

// Per-image slot of the workspace (device pointers into one big allocation).
struct NqSlot {
  const uint32_t* in;      // ARGB source pixels (device)
  uint32_t* out;           // ARGB result pixels (device)
  // histogram accumulators
  unsigned int* hCnt;              // [65536]
  unsigned long long* hSum;        // [4][65536] a,r,g,b (RGB only)
  // LAB strict-order histogram scratch
  unsigned int* keyOff;            // [65536+1] exclusive scan of hCnt
  uint32_t* sortA;                 // [npix] pixels ordered by (low byte of key)
  uint32_t* sortB;                 // [npix] pixels ordered by key, stable
  unsigned int* warpHist;          // [nRuns][256] per-run digit counts
  float* sal;                      // [npix] saliency map (PL:155-156, 499-508)
  // compacted bins (SoA). RGB uses the double arrays, LAB the float ones.
  double* bAc; double* bC1; double* bC2; double* bC3;   // means: alpha, r|L, g|A, b|B
  float* fAc; float* fC1; float* fC2; float* fC3;
  float* bCnt; float* bErr;
  int* bNn; int* bTm; int* bMtm;
  // heap (see HeapView in nq_pnn.cuh)
  uint2* heap;                     // [65538] global spill of the lower heap levels: {err bits, id | nn << 16}
  int* mergeLog;                   // optional [2*65536] (tb, nb) pairs for parity tests
  // dither
  const uint32_t* order;           // [npix] Gilbert visiting order of the image's size, x | y << 16 (shared by equal sizes)
  unsigned short* memo;            // [65536] nearestMap for reduced keys (0xFFFF = absent)
  unsigned short* idx;             // [npix] palette indices of pass 1 when a second pass follows
  unsigned char* cells;            // [32768][32] candidate lists of the CIELAB closest-colour scan (k_build_cells)
  unsigned int* bits;              // [2^27] one bit per ARGB colour ever passed to getLab (pixelMap, PL:34-42); only when the
                                   // BlueNoise second pass needs pixelMap.size() (PL:511-513)
};
