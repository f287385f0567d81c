// nq_index.h -- palette index of an output pixel (the index-map entry points, include/nquant_b200.h): the table k_index_map
// (nq_api.cu) builds in shared memory and looks every pixel up in, written once for the device and the host so that g++
// tests the same build and lookup on the CPU.
//
// The index of a pixel is the LOWEST palette index whose colour equals the output pixel, so palette[index] == argb_out
// always holds. With distinct palette colours (every palette the quantizers are known to produce) that is the index the
// reference's lookup chose. Colours are whole 0xAARRGGBB words: two entries that differ in alpha only are two colours.
#pragma once
#include <stdint.h>
#include "nq_math.h"   // NQ_HD

// Open addressing with linear probing over 1024 slots: a palette holds at most 256 colours, so the table is at most a
// quarter full and a lookup rarely probes past its first slot. A slot holds colour << 32 | index; the empty marker is no
// entry, since an entry's low word is an index below 256.
#define NQ_IMAP_SLOTS 1024
#define NQ_IMAP_EMPTY 0xFFFFFFFFFFFFFFFFULL

namespace nq {

NQ_HD unsigned imap_hash(uint32_t c) { return (c * 0x9E3779B1u) >> 22; }   // top 10 bits of a Fibonacci hash

// Entry t (0 <= t < palette length) of the table: pal[t] goes in unless an earlier entry has the same colour, so the lowest
// index wins. The table starts all NQ_IMAP_EMPTY. The colours that go in are distinct, so the table does not depend on the
// order of the inserts: on the device every thread of a block inserts entries of its own, claiming slots with atomicCAS.
NQ_HD void imap_insert(unsigned long long* tab, const uint32_t* pal, int t) {
  const uint32_t c = pal[t];
  for (int j = 0; j < t; ++j)
    if (pal[j] == c) return;
  const unsigned long long e = ((unsigned long long)c << 32) | (unsigned)t;
  for (unsigned h = imap_hash(c);; h = (h + 1) & (NQ_IMAP_SLOTS - 1)) {
#ifdef __CUDA_ARCH__
    if (atomicCAS(&tab[h], NQ_IMAP_EMPTY, e) == NQ_IMAP_EMPTY) return;
#else
    if (tab[h] == NQ_IMAP_EMPTY) { tab[h] = e; return; }
#endif
  }
}

// palette index of colour c, or -1 when the palette does not hold it
NQ_HD int imap_lookup(const unsigned long long* tab, uint32_t c) {
  for (unsigned h = imap_hash(c);; h = (h + 1) & (NQ_IMAP_SLOTS - 1)) {
    const unsigned long long e = tab[h];
    if (e == NQ_IMAP_EMPTY) return -1;
    if ((uint32_t)(e >> 32) == c) return (int)(uint32_t)e;
  }
}

}  // namespace nq
