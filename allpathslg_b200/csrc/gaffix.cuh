// gaffix.cuh -- device side of the affixes on the sharded table (apgk_group_build_affixes, include/apgk.h; host side
// in group.cuh).  Each rank's reads hold windows of k-mers every rank owns, so every window's affix byte travels to
// the k-mer's owner, on the query exchange of the frequency lookups (gfreq.cuh).  Per batch of a rank's read store,
//   sender  k_occ_scatter (histogram mode) by coarse bucket, then k_aff_scatter (affix.cuh) over the batch's base
//           range: every window's level-1 element and affix byte into B, bucket-major.  4-byte remainders: one u64 per
//           slot (rem << 8 | affix); full keys: the key at slot i, the byte at slot i of a byte plane in the same B
//   all     the bucket sizes all-gathered and scanned into per-source piece offsets, as in the lookups
//   owner   k_gaff_place: one CTA per owned coarse bucket, reading every source's piece over peer memory and ORing
//           the bytes into its own affix array.  Nothing goes back to the sender: the owner only reads peer memory.
#pragma once
#include "affix.cuh"
#include "gfreq.cuh"

namespace apgk {

struct GaffArgs {
  const void* const* src;                 // [n_src] the senders' partition buffers B (peer memory)
  const unsigned long long* plane_off;    // [n_src] byte offset of each sender's affix-byte plane in its B (full keys)
  const unsigned long long* piece_off;    // [n_src][nb + 1] first slot of each sender's piece of each bucket
  uint32_t n_src, nb, me, lo, hi;         // this CTA grid places the owned coarse buckets [lo, hi)
  int d2, rem_bits, pad;                  // shard index = coarse bucket << d2; rem_bits / pad of the partition geometry
  uint32_t* aff32;                        // the shard's affix bytes as aligned u32 words (zeroed before the first batch)
  unsigned long long* counters;           // [0] elements whose k-mer is not in the table (must stay 0), [1] elements from peers
};

// The shard's table slice of the bucket sits in shared memory as sorted remainders with a packed per-row byte array
// (4-byte remainders and slices of at most GF_CAP keys); every element finds its row by binary search and ORs its
// byte there, then the rows go out as atomicOr on aligned u32 words (neighbouring buckets share words).  Full keys
// and larger slices search the shard's table in global memory and OR into the affix array directly.
template <int W, typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_gaff_place(FreqTable<W> t, GaffArgs a) {
  constexpr bool U32 = sizeof(Elem) == 4;
  __shared__ uint32_t sh_rem[U32 ? GF_CAP : 1], sh_aff[U32 ? GF_CAP / 4 : 1];
  unsigned long long missing = 0, remote = 0;
  for (uint32_t b = a.lo + blockIdx.x; b < a.hi; b += gridDim.x) {
    // a bucket no source sent anything to this batch is skipped: its slice is not loaded (the same on every thread)
    unsigned long long n_all = 0;
    for (uint32_t s = 0; s < a.n_src; s++) {
      const unsigned long long* po = a.piece_off + (size_t)s * ((size_t)a.nb + 1);
      n_all += po[b + 1] - po[b];
    }
    if (!n_all) continue;
    const unsigned long long t0 = t.index[(size_t)b << a.d2], d = t.index[(size_t)(b + 1) << a.d2] - t0;
    bool in_sh = false;
    if constexpr (U32) {
      in_sh = d <= GF_CAP;
      if (in_sh) {
        for (uint32_t j = threadIdx.x; j < (uint32_t)d; j += NT) sh_rem[j] = OccElem<Elem, W>::make(t.keys[t0 + j], a.rem_bits, a.pad);
        for (uint32_t j = threadIdx.x; j < ((uint32_t)d + 3) / 4; j += NT) sh_aff[j] = 0;
        __syncthreads();
      }
    }
    for (uint32_t s = 0; s < a.n_src; s++) {
      const unsigned long long* po = a.piece_off + (size_t)s * ((size_t)a.nb + 1);
      const unsigned long long e0 = po[b], n = po[b + 1] - e0;
      if (s != a.me) remote += n;
      for (unsigned long long i = threadIdx.x; i < n; i += NT) {
        Key<W> c;
        uint32_t v;
        if constexpr (U32) {
          const unsigned long long x = static_cast<const unsigned long long*>(a.src[s])[e0 + i];
          const uint32_t r = (uint32_t)(x >> 8);
          v = (uint32_t)x & 0xFFu;
          if (in_sh) {
            uint32_t lo = 0, hi = (uint32_t)d;
            while (lo < hi) {
              const uint32_t mid = (lo + hi) >> 1;
              if (sh_rem[mid] < r) lo = mid + 1; else hi = mid;
            }
            if (lo < (uint32_t)d && sh_rem[lo] == r) {
              if (v) atomicOr(&sh_aff[lo >> 2], v << (8u * (lo & 3u)));
            } else {
              missing++;
            }
            continue;
          }
          c = OccElem<Elem, W>::key(r, b, a.rem_bits, a.pad);
        } else {
          c = static_cast<const Key<W>*>(a.src[s])[e0 + i];
          v = static_cast<const uint8_t*>(a.src[s])[a.plane_off[s] + e0 + i];
        }
        const unsigned long long idx = table_find_index(t, c);
        if (idx == ~0ull) missing++;
        else aff_or_byte(a.aff32, idx, v);
      }
    }
    if (in_sh) {
      __syncthreads();
      // write-out: global words [t0 >> 2, (t0 + d - 1) >> 2], each assembled from the shared bytes of its rows
      const unsigned long long w0 = t0 >> 2, w1 = (t0 + d + 3) >> 2;
      for (unsigned long long w = w0 + threadIdx.x; w < w1; w += NT) {
        uint32_t v = 0;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) {
          const unsigned long long row = 4 * w + k;
          if (row >= t0 && row < t0 + d) {
            const uint32_t j = (uint32_t)(row - t0);
            v |= ((sh_aff[j >> 2] >> (8u * (j & 3u))) & 0xFFu) << (8u * k);
          }
        }
        if (v) atomicOr(&a.aff32[w], v);
      }
      __syncthreads();   // the slice is reloaded for the next bucket
    }
  }
  if (missing) atomicAdd(&a.counters[0], missing);
  if (threadIdx.x == 0 && remote) atomicAdd(&a.counters[1], remote);
}

// counters[3] += *n: the windows a sender placed in this batch (the last entry of its piece offsets)
__global__ void k_gaff_sent(const unsigned long long* __restrict__ n, unsigned long long* __restrict__ counters) {
  counters[3] += *n;
}

}  // namespace apgk
