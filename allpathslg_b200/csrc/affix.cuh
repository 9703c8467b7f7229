// affix.cuh -- k-mer AFFIXES: for every distinct canonical k-mer of the sorted table, which of the four bases
// precede it and which follow it somewhere in the reads (one byte: bit b = base b precedes, bit 4+b = base b
// follows, in the canonical orientation).  What the unipath / graph code reads per k-mer: the naif_kmer
// "k-mer + frequency + affixes" record (KmerFreqAffixes [U]; SURVEY.md's recollection, no file:line exists).
// The contract, palindromes included, is stated in include/apgk.h.
//
// B200 formulation: the two-phase shape of the occurrence records (occ.cuh), with a 1-byte payload:
//   k_aff_scatter: one sweep over the read store; every valid window sends its level-1 element and its affix
//               byte to ITS prefix bucket's region (bucket regions: occ_run_offsets + k_occ_bstart).  The
//               neighbour bases come from the words the extraction already holds, their existence from the
//               start bitmap.  u32 remainders: one u64 per window (rem << 8 | affix); full keys: the key plus a
//               byte array.  No position is stored.
//   k_aff_place: one CTA per bucket; the bucket's keys sit in shared memory as sorted remainders, each element
//               finds its row by binary search and ORs its byte into a shared per-row byte (packed in u32 words);
//               the bucket's bytes then go out sequentially.  Full keys and buckets beyond the shared table
//               search the table in global memory.
// Every global update of the affix array is an atomicOr on an aligned u32 word (two buckets' rows can share a
// word), on an array zeroed first: the result does not depend on scheduling.
#pragma once
#include "occ.cuh"

namespace apgk {

// reverse the order of the 4 bits of a base mask: bit b -> bit 3-b (the complement of every base)
APGK_HD uint32_t aff_comp4(uint32_t m) { return ((m & 1u) << 3) | ((m & 2u) << 1) | ((m & 4u) >> 1) | ((m & 8u) >> 3); }

// Affix byte of a k-mer -> affix byte of its reverse complement: pre' = comp(suf), suf' = comp(pre).
APGK_HD uint32_t aff_revcomp(uint32_t a) { return aff_comp4((a >> 4) & 15u) | (aff_comp4(a & 15u) << 4); }

// OR `a` into byte `i` of a byte array viewed as aligned u32 words
__device__ __forceinline__ void aff_or_byte(uint32_t* __restrict__ aff32, unsigned long long i, uint32_t a) {
  if (a) atomicOr(&aff32[i >> 2], a << (8u * (uint32_t)(i & 3)));
}

// Sweep of the reads: every valid window takes the next slot of its prefix bucket and stores its element with
// its affix byte there.  U32 elements: elem64[o] = rem << 8 | affix.  Full keys: keys[o] = key, bytes[o] = affix.
// Only the windows starting in [first, first + n_bases) take part (the whole store on one GPU, a batch of it in the
// group build, gaffix.cuh); their neighbours are read from the store itself, so a batch's edges change no byte.
template <int W, typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_aff_scatter(ReadStore rs, FreqTable<W> t, uint64_t first, uint64_t n_bases,
                                                    unsigned long long* __restrict__ bcur,
                                                    unsigned long long* __restrict__ elem64, Key<W>* __restrict__ keys,
                                                    uint8_t* __restrict__ bytes, unsigned long long n_slots,
                                                    unsigned long long* __restrict__ counters) {
  constexpr bool U32 = sizeof(Elem) == 4;
  const uint64_t p = (first & ~15ull) + ((uint64_t)blockIdx.x * NT + threadIdx.x) * POS_PER_THREAD;
  const uint64_t end = first + n_bases;
  if (p >= end) return;
  uint32_t valid = window_valid_mask16(rs.starts32, p, rs.K, rs.total_bases);
  if (p < first) valid &= 0xFFFFu << (uint32_t)(first - p);
  if (end - p < 16) valid &= (1u << (uint32_t)(end - p)) - 1u;
  if (!valid) return;
  Window16<W> win;
  load_window16<W>(rs.bases32, p, rs.K, win);
  // neighbours: base p+j-1 precedes window j (base p-1 for j = 0), base p+j+K follows it (win.v0)
  const uint32_t prev = p ? (rs.bases32[(p >> 4) - 1] >> 30) : 0u;
  // a neighbour exists when its read did not start at the window (left) / at the base after it (right)
  const uint32_t st_l = rs.starts32[p >> 5] >> (uint32_t)(p & 31);           // bit j: a read starts at p+j
  const uint64_t q = p + (uint64_t)rs.K;
  const uint32_t st_r = funnel_r(rs.starts32[q >> 5], rs.starts32[(q >> 5) + 1], (uint32_t)(q & 31));  // bit j: at p+j+K
  const bool even_k = (rs.K & 1) == 0;
  extract16<W>(win, rs.K, [&](int j, const Key<W>& c, bool use_rc) {
    if ((valid >> j) & 1u) {
      uint32_t a = 0;
      if (!((st_l >> j) & 1u) && p + (uint64_t)j > 0) a |= 1u << (j ? (win.w[0] >> (2 * (j - 1))) & 3u : prev);
      if (!((st_r >> j) & 1u) && q + (uint64_t)j < rs.total_bases) a |= 16u << ((win.v0 >> (2 * j)) & 3u);
      if (use_rc) {
        a = aff_revcomp(a);
      } else if (even_k && key_eq(c, key_revcomp(c, rs.K))) {
        a |= aff_revcomp(a);   // a palindrome is its own reverse complement: both readings apply
      }
      const uint32_t b = digit_of(c, t.prefix_pos, t.prefix_len, t.pad);
      const unsigned long long o = atomicAdd(&bcur[b], 1ull);
      if (o >= n_slots) {
        atomicAdd(&counters[2], 1ull);
      } else if constexpr (U32) {
        elem64[o] = ((unsigned long long)OccElem<Elem, W>::make(c, t.prefix_pos, t.pad) << 8) | a;
      } else {
        keys[o] = c;
        bytes[o] = (uint8_t)a;
      }
    }
  });
}

// One CTA per prefix bucket (grid-stride): OR every element's affix byte into its k-mer's row of aff32
// (n_distinct bytes, zeroed).  counters[1] counts elements whose k-mer is missing from the table.
template <int W, typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_aff_place(FreqTable<W> t, const unsigned long long* __restrict__ bstart,
                                                  const unsigned long long* __restrict__ elem64,
                                                  const Key<W>* __restrict__ keys, const uint8_t* __restrict__ bytes,
                                                  uint32_t* __restrict__ aff32, unsigned long long* __restrict__ counters) {
  constexpr bool U32 = sizeof(Elem) == 4;
  __shared__ uint32_t sh_rem[U32 ? OCC_PLACE_CAP : 1], sh_aff[U32 ? OCC_PLACE_CAP / 4 : 1];
  for (uint32_t b = blockIdx.x; b < t.nb; b += gridDim.x) {
    const unsigned long long e0 = bstart[b], n = bstart[b + 1] - e0;
    if (!n) continue;
    const unsigned long long t0 = t.index[b], d = t.index[b + 1] - t0;
    if (U32 && d <= OCC_PLACE_CAP) {
      if constexpr (U32) {
        for (uint32_t j = threadIdx.x; j < (uint32_t)d; j += NT) {
          sh_rem[j] = OccElem<Elem, W>::make(t.keys[t0 + j], t.prefix_pos, t.pad);
          if ((j & 3) == 0) sh_aff[j >> 2] = 0;
        }
        __syncthreads();
        unsigned long long missing = 0;
        for (unsigned long long i = threadIdx.x; i < n; i += NT) {
          const unsigned long long v = elem64[e0 + i];
          const uint32_t r = (uint32_t)(v >> 8);
          uint32_t lo = 0, hi = (uint32_t)d;
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (sh_rem[mid] < r) lo = mid + 1; else hi = mid;
          }
          if (lo < (uint32_t)d && sh_rem[lo] == r) {
            const uint32_t a = (uint32_t)v & 0xFFu;
            if (a) atomicOr(&sh_aff[lo >> 2], a << (8u * (lo & 3u)));
          } else {
            missing++;
          }
        }
        if (missing) atomicAdd(&counters[1], missing);
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
          if (v) atomicOr(&aff32[w], v);
        }
        __syncthreads();   // the shared table is reloaded for the next bucket
      }
    } else {
      unsigned long long missing = 0;
      for (unsigned long long i = threadIdx.x; i < n; i += NT) {
        Key<W> c;
        uint32_t a;
        if constexpr (U32) {
          const unsigned long long v = elem64[e0 + i];
          c = OccElem<Elem, W>::key((uint32_t)(v >> 8), b, t.prefix_pos, t.pad);
          a = (uint32_t)v & 0xFFu;
        } else {
          c = keys[e0 + i];
          a = bytes[e0 + i];
        }
        const unsigned long long idx = table_find_index(t, c);
        if (idx == ~0ull) missing++;
        else aff_or_byte(aff32, idx, a);
      }
      if (missing) atomicAdd(&counters[1], missing);
    }
  }
}

// Affixes (and counts) of arbitrary k-mers, in the QUERY's orientation: a query that is the reverse complement of
// its canonical form gets the transformed byte.  Absent k-mers: affixes 0, count 0.
template <int W>
__global__ void k_lookup_affixes(FreqTable<W> t, const uint8_t* __restrict__ aff, const Key<W>* __restrict__ q, uint64_t nq,
                                 int K, int canonicalise, uint8_t* __restrict__ aff_out, uint32_t* __restrict__ cnt_out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  Key<W> c = q[i];
  bool rev = false;
  if (canonicalise) {
    const Key<W> rc = key_revcomp(c, K);
    rev = key_less(rc, c);
    if (rev) c = rc;
  }
  const unsigned long long idx = table_find_index(t, c);
  uint32_t a = 0, n = 0;
  if (idx != ~0ull) {
    a = aff[idx];
    n = t.counts[idx];
    if (rev) a = aff_revcomp(a);
  }
  aff_out[i] = (uint8_t)a;
  cnt_out[i] = n;
}

}  // namespace apgk
