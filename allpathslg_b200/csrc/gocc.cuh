// gocc.cuh -- device side of the occurrence records on the sharded table (apgk_group_build_occurrences,
// include/apgk.h; host side in group.cuh).  Each rank's reads hold windows of k-mers every rank owns, so every
// window's record travels to the k-mer's owner, on the query exchange of the frequency lookups (gfreq.cuh).  An owner
// cannot turn a base position of another rank's store into a read id (it lacks that rank's start bitmap), so the
// sender does, and the record arrives in its final form
//   (group read id << 32) | ((position in read - 1) << 1) | canonical_is_reverse
// whose ascending u64 order is ascending (read id, position), as on one GPU.  Per batch of a rank's read store,
//   sender  k_occ_scatter (histogram mode) by coarse bucket, then k_gocc_scatter over the batch's base range: every
//           window's level-1 element into B, bucket-major, its record at the same slot of a u64 plane in the same B
//   all     the bucket sizes all-gathered and scanned into per-source piece offsets, as in the lookups
//   owner   k_gocc_place: one CTA per owned coarse bucket, reading every source's piece over peer memory; each record
//           takes the next slot of its k-mer's run in the shard's own record array.  Nothing goes back to the sender.
// After the last batch k_occ_sort_small / k_occ_sort_big (occ.cuh) sort every run; the records are unique, so the
// result does not depend on the batches, the world size or the order of the atomics.
#pragma once
#include "gfreq.cuh"

namespace apgk {

struct GoccReads {                        // what the sweep needs to number the reads of its store
  const unsigned long long* blk_rank;     // rank directory over the start bitmap (k_start_blocks + scan)
  const unsigned long long* empty_nb;     // [n_empty] reads without bases (occ_read_id)
  uint32_t n_empty;
  unsigned long long read_base;           // group read id of the store's first read: the reads of the ranks before it
};

// Sweep of the batch [first, first + n_bases): every valid window takes the next slot of its coarse bucket and stores
// its element at elems[o] and its record at recs[o].  The read of the thread's first valid window comes from the rank
// directory; its other windows count the read starts between (the 16 positions share one start word).
template <int W, typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_gocc_scatter(ReadStore rs, FreqTable<W> t, uint64_t first, uint64_t n_bases,
                                                     unsigned long long* __restrict__ bcur, Elem* __restrict__ elems,
                                                     unsigned long long* __restrict__ recs, unsigned long long n_slots,
                                                     GoccReads rd, unsigned long long* __restrict__ counters) {
  const uint64_t p = (first & ~15ull) + ((uint64_t)blockIdx.x * NT + threadIdx.x) * POS_PER_THREAD;
  const uint64_t end = first + n_bases;
  if (p >= end) return;
  uint32_t valid = window_valid_mask16(rs.starts32, p, rs.K, rs.total_bases);
  if (p < first) valid &= 0xFFFFu << (uint32_t)(first - p);
  if (end - p < 16) valid &= (1u << (uint32_t)(end - p)) - 1u;
  if (!valid) return;
  const uint32_t j0 = (uint32_t)__ffs((int)valid) - 1u;
  unsigned long long rank0;
  uint64_t s0;
  occ_start_rank(rs.starts32, rd.blk_rank, p + j0, rank0, s0);
  const uint32_t st = (rs.starts32[p >> 5] >> (uint32_t)(p & 31)) & 0xFFFFu;   // bit j: a read starts at p + j
  Window16<W> win;
  load_window16<W>(rs.bases32, p, rs.K, win);
  extract16<W>(win, rs.K, [&](int j, const Key<W>& c, bool use_rc) {
    if ((valid >> j) & 1u) {
      const uint32_t later = st & ((2u << j) - 1u) & ~((2u << j0) - 1u);   // read starts in (p + j0, p + j]
      const uint64_t s = later ? p + (31u - (uint32_t)__clz((int)later)) : s0;
      const unsigned long long id = rd.read_base + occ_read_id(rank0 + (uint32_t)__popc(later), rd.empty_nb, rd.n_empty);
      const unsigned long long rec = (id << 32) | ((p + (uint64_t)j - s) << 1) | (use_rc ? 1ull : 0ull);
      const uint32_t b = digit_of(c, t.prefix_pos, t.prefix_len, t.pad);
      const unsigned long long o = atomicAdd(&bcur[b], 1ull);
      if (o >= n_slots) {
        atomicAdd(&counters[2], 1ull);
      } else {
        elems[o] = OccElem<Elem, W>::make(c, t.prefix_pos, t.pad);
        recs[o] = rec;
      }
    }
  });
}

struct GoccArgs {
  const void* const* src;                 // [n_src] the senders' partition buffers B (peer memory)
  const unsigned long long* plane_off;    // [n_src] byte offset of each sender's record plane in its B
  const unsigned long long* piece_off;    // [n_src][nb + 1] first slot of each sender's piece of each bucket
  uint32_t n_src, nb, me, lo, hi;         // this CTA grid places the owned coarse buckets [lo, hi)
  int d2, rem_bits, pad;                  // shard index = coarse bucket << d2; rem_bits / pad of the partition geometry
  const unsigned long long* run_off;      // [D + 1] the shard's run offsets
  uint32_t* cursor;                       // [D] slots of each run filled so far (zeroed before the first batch)
  unsigned long long* occ;                // the shard's records
  unsigned long long* counters;           // [0] elements whose k-mer is not in the table, [1] elements from peers,
                                          // [2] slots past a bucket (sweep) or past a run (here): both must stay 0
};

// 4-byte remainders of a slice of at most OCC_PLACE_CAP keys whose runs span fewer than 2^32 slots: the slice's
// remainders, its run offsets relative to the slice's first slot and the rows' cursors sit in shared memory; every
// element finds its row by binary search there and takes a slot with a shared atomic, warp after warp (the runs
// then receive each piece in element order, nearly sorted), and the cursors go back to global memory for the next
// batch.  Full keys and other slices search the shard's table in global memory and take a slot with a global atomic.
template <int W, typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_gocc_place(FreqTable<W> t, GoccArgs a) {
  constexpr bool U32 = sizeof(Elem) == 4;
  constexpr uint32_t NONE = 0xFFFFFFFFu;
  __shared__ uint32_t sh_rem[U32 ? OCC_PLACE_CAP : 1], sh_off[U32 ? OCC_PLACE_CAP + 1 : 1], sh_cur[U32 ? OCC_PLACE_CAP : 1];
  unsigned long long missing = 0, past = 0, remote = 0;
  for (uint32_t b = a.lo + blockIdx.x; b < a.hi; b += gridDim.x) {
    // a bucket no source sent anything to this batch is skipped (the same on every thread)
    unsigned long long n_all = 0;
    for (uint32_t s = 0; s < a.n_src; s++) {
      const unsigned long long* po = a.piece_off + (size_t)s * ((size_t)a.nb + 1);
      n_all += po[b + 1] - po[b];
    }
    if (!n_all) continue;
    const unsigned long long t0 = t.index[(size_t)b << a.d2], d = t.index[(size_t)(b + 1) << a.d2] - t0;
    const unsigned long long e0 = a.run_off[t0];   // first slot of the slice's runs
    bool in_sh = false;
    if constexpr (U32) {
      in_sh = d <= OCC_PLACE_CAP && a.run_off[t0 + d] - e0 < (1ull << 32);
      if (in_sh) {
        for (uint32_t j = threadIdx.x; j <= (uint32_t)d; j += NT) {
          sh_off[j] = (uint32_t)(a.run_off[t0 + j] - e0);
          if (j < (uint32_t)d) {
            sh_rem[j] = OccElem<Elem, W>::make(t.keys[t0 + j], a.rem_bits, a.pad);
            sh_cur[j] = a.cursor[t0 + j];
          }
        }
        __syncthreads();
      }
    }
    for (uint32_t s = 0; s < a.n_src; s++) {
      const unsigned long long* po = a.piece_off + (size_t)s * ((size_t)a.nb + 1);
      const unsigned long long p0 = po[b], n = po[b + 1] - p0;
      if (s != a.me) remote += n;
      const Elem* el = static_cast<const Elem*>(a.src[s]) + p0;
      const unsigned long long* rec =
          reinterpret_cast<const unsigned long long*>(static_cast<const uint8_t*>(a.src[s]) + a.plane_off[s]) + p0;
      if (in_sh) {
        if constexpr (U32) {
          for (unsigned long long i0 = 0; i0 < n; i0 += NT) {
            const unsigned long long i = i0 + threadIdx.x;
            uint32_t row = NONE;
            unsigned long long v = 0;
            if (i < n) {
              const uint32_t r = el[i];
              v = rec[i];
              uint32_t lo = 0, hi = (uint32_t)d;
              while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (sh_rem[mid] < r) lo = mid + 1; else hi = mid;
              }
              if (lo < (uint32_t)d && sh_rem[lo] == r) row = lo; else missing++;
            }
#pragma unroll 1
            for (int w = 0; w < NT / 32; w++) {
              if ((int)(threadIdx.x >> 5) == w && row != NONE) {
                const uint32_t slot = sh_off[row] + atomicAdd(&sh_cur[row], 1u);
                if (slot < sh_off[row + 1]) a.occ[e0 + slot] = v; else past++;
              }
              __syncthreads();
            }
          }
        }
      } else {
        for (unsigned long long i = threadIdx.x; i < n; i += NT) {
          const unsigned long long idx = table_find_index(t, OccElem<Elem, W>::key(el[i], b, a.rem_bits, a.pad));
          if (idx == ~0ull) {
            missing++;
          } else {
            const unsigned long long o = a.run_off[idx] + atomicAdd(&a.cursor[idx], 1u);
            if (o < a.run_off[idx + 1]) a.occ[o] = rec[i]; else past++;
          }
        }
      }
    }
    if (in_sh) {
      __syncthreads();
      for (uint32_t j = threadIdx.x; j < (uint32_t)d; j += NT) a.cursor[t0 + j] = sh_cur[j];
      __syncthreads();   // the slice is reloaded for the next bucket
    }
  }
  if (missing) atomicAdd(&a.counters[0], missing);
  if (past) atomicAdd(&a.counters[2], past);
  if (threadIdx.x == 0 && remote) atomicAdd(&a.counters[1], remote);
}

// a shard's records -> read_id[i], pos[i] (1-based, negative when the canonical form is the reverse complement)
__global__ void k_gocc_decode(const unsigned long long* __restrict__ occ, uint64_t n, uint32_t* __restrict__ read_id,
                              int32_t* __restrict__ pos) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long v = occ[i];
  const int32_t p1 = (int32_t)((v >> 1) & 0x7FFFFFFFull) + 1;
  read_id[i] = (uint32_t)(v >> 32);
  pos[i] = (v & 1ull) ? -p1 : p1;
}

}  // namespace apgk
