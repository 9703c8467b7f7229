// gfreq.cuh -- device side of the frequency lookups on the sharded table (apgk_group_read_freqs_device,
// include/apgk.h; host side in group.cuh).  After apgk_group_count every rank holds the table of the k-mers it
// OWNS, but its reads contain k-mers owned by every rank.  The queries travel to the owner, not the table to the
// queries: per batch of a rank's base range,
//   sender  k_occ_scatter (occ.cuh), twice: bucket histogram of the P-bit canonical prefix, then every window's
//           level-1 element into B (the exported partition buffer) in bucket-major order, its batch-relative
//           position (u32) at the same slot of a local array
//   all     the bucket sizes all-gathered and scanned into per-source piece offsets, as in the count
//   owner   k_gf_resolve: one CTA per owned bucket; the shard's table slice of the bucket sits in shared memory
//           (remainders + counts), the CTA reads every source's piece of the bucket straight from the source's B
//           over peer memory and writes the count IN PLACE over each query
//   sender  k_gf_scatter: out[pos[slot]] = the count now in B[slot]
#pragma once
#include "occ.cuh"

namespace apgk {

constexpr int GF_NT = 256;
constexpr uint32_t GF_CAP = 4096;   // table keys of one bucket the shared-memory slice holds (remainder + count: 32 KB)

template <typename Elem>
struct GfArgs {
  Elem* const* src;                       // [n_src] the senders' partition buffers (peer memory): queries, bucket-major
  const unsigned long long* piece_off;    // [n_src][nb + 1] first slot of each sender's piece of each bucket
  uint32_t n_src, nb, me, lo, hi;         // this CTA grid resolves the owned coarse buckets [lo, hi)
  int d2, rem_bits, pad;                  // shard index = coarse bucket << d2; rem_bits / pad of the partition geometry
  unsigned long long* counters;           // [0] queries whose k-mer is not in the table (must stay 0), [1] queries from peers;
                                          // [2] slots past a bucket (k_occ_scatter), [3] queries resolved (k_gf_scatter)
};

// The count of a query is written over the first 4 bytes of its slot: a 32-bit remainder is replaced, a full key
// keeps its other words.  Full-key elements (and slices above GF_CAP keys) search the shard's table in global
// memory with table_find_index; both paths give the same count.
template <int W, typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_gf_resolve(FreqTable<W> t, GfArgs<Elem> a) {
  constexpr bool U32 = sizeof(Elem) == 4;
  __shared__ uint32_t sh_rem[U32 ? GF_CAP : 1], sh_cnt[U32 ? GF_CAP : 1];
  unsigned long long missing = 0, remote = 0;
  for (uint32_t b = a.lo + blockIdx.x; b < a.hi; b += gridDim.x) {
    const unsigned long long t0 = t.index[(size_t)b << a.d2], d = t.index[(size_t)(b + 1) << a.d2] - t0;
    bool in_sh = false;
    if constexpr (U32) {
      in_sh = d <= GF_CAP;
      if (in_sh) {
        for (uint32_t j = threadIdx.x; j < (uint32_t)d; j += NT) {
          sh_rem[j] = OccElem<Elem, W>::make(t.keys[t0 + j], a.rem_bits, a.pad);
          sh_cnt[j] = t.counts[t0 + j];
        }
        __syncthreads();
      }
    }
    for (uint32_t s = 0; s < a.n_src; s++) {
      const unsigned long long* po = a.piece_off + (size_t)s * ((size_t)a.nb + 1);
      const unsigned long long e0 = po[b], n = po[b + 1] - e0;
      if (s != a.me) remote += n;
      Elem* q = a.src[s] + e0;
      for (unsigned long long i = threadIdx.x; i < n; i += NT) {
        const Elem e = q[i];
        uint32_t cnt = 0;
        bool found = false;
        if (in_sh) {
          if constexpr (U32) {
            uint32_t lo = 0, hi = (uint32_t)d;
            while (lo < hi) {
              const uint32_t mid = (lo + hi) >> 1;
              if (sh_rem[mid] < e) lo = mid + 1; else hi = mid;
            }
            found = lo < (uint32_t)d && sh_rem[lo] == e;
            if (found) cnt = sh_cnt[lo];
          }
        } else {
          const unsigned long long idx = table_find_index(t, OccElem<Elem, W>::key(e, b, a.rem_bits, a.pad));
          found = idx != ~0ull;
          if (found) cnt = t.counts[idx];
        }
        if (!found) missing++;
        reinterpret_cast<uint32_t*>(q + i)[0] = cnt;
      }
    }
    if (in_sh) __syncthreads();   // the slice is reloaded for the next bucket
  }
  if (missing) atomicAdd(&a.counters[0], missing);
  if (threadIdx.x == 0 && remote) atomicAdd(&a.counters[1], remote);
}

// out[pos[i]] = count in slot i, for the *n_slots slots of this batch; counters[3] += *n_slots (queries resolved)
template <typename Elem>
__global__ void k_gf_scatter(const Elem* __restrict__ B, const uint32_t* __restrict__ pos, const unsigned long long* __restrict__ n_slots,
                             uint32_t* __restrict__ out, unsigned long long* __restrict__ counters) {
  const unsigned long long n = *n_slots;
  if (blockIdx.x == 0 && threadIdx.x == 0) counters[3] += n;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
    out[pos[i]] = reinterpret_cast<const uint32_t*>(B + i)[0];
}

}  // namespace apgk
