// Remap oracle (test infrastructure): the reference's convert(nMaxColors, dither) with the palette the dither receives
// replaced by the caller's, i.e. PnnQuantizer.java:409-456 / PnnLABQuantizer.java:492-522 with dither(...) called on
// another palette. It derives from the oracle's quantizers (oracle/nq_oracle.cpp, included unchanged) and overrides two
// protected hooks only:
//  - ditherImage: every branch of convert (pnnquan's palette, the few-colours return of PL:193-206, the fixed palette of
//    PQ:441-452) hands its palette to ditherImage, which dithers to the caller's palette instead;
//  - pnnquan: runs in full, so every member the dither reads (weight, PR/PG/PB/PA, ratio after its re-tune, isNano,
//    saliencies, pixelMap) is what convert leaves. The merge loop and the palette fill after the re-tune of ratio write
//    none of those members; a palette fill that throws (ColorUtils.setAlphaComponent, CIELABConvertor.java:79) does so
//    after all of them are set, and its palette is discarded anyway, so the remap goes on.
#include "../oracle/nq_oracle.cpp"

namespace {
template <class Q>
class Remapper : public Q {
 public:
  std::vector<int32_t> callerPalette;
  Remapper(const uint32_t* argb, int w, int h) : Q(argb, w, h) {}

 protected:
  std::vector<int32_t> pnnquan(const std::vector<int32_t>& pixels, int nMaxColors) override {
    try {
      return Q::pnnquan(pixels, nMaxColors);
    } catch (const std::invalid_argument&) {
      return callerPalette;
    }
  }
  std::vector<int32_t> ditherImage(const std::vector<int32_t>& cPixels, std::vector<int32_t>& palette, int width, int height,
                                   bool dither) override {
    return Q::ditherImage(cPixels, callerPalette, width, height, dither);
  }
};

template <class Q>
int run_remap(nqo_handle* h, const uint32_t* argb, int w, int hgt, int nMaxColors, int dither, uint64_t seed, const uint32_t* palette,
              int palette_len, uint32_t* out) {
  Remapper<Q> q(argb, w, hgt);
  q.rngSeed = seed;
  q.callerPalette.assign(reinterpret_cast<const int32_t*>(palette), reinterpret_cast<const int32_t*>(palette) + palette_len);
  const std::vector<int32_t> o = q.convert(nMaxColors, dither != 0);
  h->trace = q.trace;
  h->palette = q.callerPalette;
  memcpy(out, o.data(), o.size() * 4);
  return 0;
}
}  // namespace

extern "C" {
// kind: 0 = PnnQuantizer, 1 = PnnLABQuantizer; the scalars of the run through nqo_get_scalars(h, ..)
int nqr_remap(nqo_handle* h, int kind, const uint32_t* argb, int w, int hgt, int nMaxColors, int dither, uint64_t seed,
              const uint32_t* palette, int palette_len, uint32_t* out) {
  try {
    M.mode = 0;
    if (kind == 0) return run_remap<PnnQuantizer>(h, argb, w, hgt, nMaxColors, dither, seed, palette, palette_len, out);
    return run_remap<PnnLABQuantizer>(h, argb, w, hgt, nMaxColors, dither, seed, palette, palette_len, out);
  } catch (const std::exception& e) {
    h->error = e.what();
    return -1;
  }
}
}
