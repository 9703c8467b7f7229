// occ.cuh -- k-mer OCCURRENCE records: for every distinct canonical k-mer of the sorted table, the
// (read id, signed position) of each of its instances.  This is the payload half of what the
// reference's builders emit (SortKmers' kmer records = k-mer + read id + signed position;
// KmerParcels' batches = k-mer + list of (read id, position) -- BASELINE.json north_star names,
// SURVEY.md section 8(a) rows 1-2 and 8(f) rank 2; no file:line available, the reference tree was empty).
//
// B200 formulation: the (k-mer, count) table already exists, so the payload is not carried through
// the partition passes (that would double their HBM traffic).  Instead
//   run_off   = exclusive scan of the counts                      (one run of slots per distinct k-mer)
//   bstart[b] = run_off[index[b]]: the slots of prefix bucket b are one contiguous region
//   k_occ_scatter: second sweep over the read store; every window goes to ITS BUCKET's region (one
//               global atomic on the bucket's cursor -- 2^P counters, L2 resident) as an element
//               (32-bit remainder or full key) plus (global base position << 1 | canonical-is-reverse)
//   k_occ_place: one CTA per bucket; the bucket's table keys sit in shared memory as sorted
//               remainders, every element finds its k-mer by binary search there, takes a slot of that
//               k-mer's run with a shared-memory atomic and writes its position -- all global traffic
//               is sequential per bucket.  Buckets with more keys than the shared table holds, and
//               full-key elements, search the table in global memory instead (same result).
//   (k_occ_fill, the first version, does lookup + slot + store straight from the sweep: every step a
//    random DRAM access, 973 ms for 4.56 G instances; kept behind APGK_OCC_DIRECT=1 as a cross-check.)
//   k_occ_sort_small / k_occ_sort_big: each run ascending by position.  The sweep visits positions
//               in ascending order, so runs arrive almost sorted: one thread per run does an
//               insertion sort that is linear on sorted input; runs above OCC_SMALL_MAX go to a
//               CTA-wide bitonic network (shared memory up to OCC_SH_CAP entries, else in place).
// The result is deterministic (independent of atomic order).  (read id, position) are derived from
// the global position on demand by k_occ_translate through a rank directory over the start bitmap.
#pragma once
#include "table.cuh"

namespace apgk {

constexpr uint32_t OCC_SMALL_MAX = 256;   // longest run one thread sorts by insertion
constexpr uint32_t OCC_SH_CAP = 4096;     // longest run the CTA sorts in shared memory (32 KB)
constexpr int OCC_BIG_NT = 512;
constexpr int RANK_BLOCK_WORDS = 8;       // rank directory granularity: 8 bitmap words = 256 bases

// counters[0] = number of big runs, counters[1] = windows whose k-mer was not in the table (must stay 0),
// counters[2] = slots beyond a run's end (must stay 0)
template <int W, int NT>
__global__ void __launch_bounds__(NT) k_occ_fill(ReadStore rs, FreqTable<W> t, const unsigned long long* __restrict__ run_off,
                                                 uint32_t* __restrict__ cursor, unsigned long long* __restrict__ occ,
                                                 unsigned long long* __restrict__ counters) {
  const uint64_t p = ((uint64_t)blockIdx.x * NT + threadIdx.x) * POS_PER_THREAD;
  if (p >= rs.total_bases) return;
  const uint32_t valid = window_valid_mask16(rs.starts32, p, rs.K, rs.total_bases);
  if (!valid) return;
  Window16<W> win;
  load_window16<W>(rs.bases32, p, rs.K, win);
  extract16<W>(win, rs.K, [&](int j, const Key<W>& c, bool use_rc) {
    if ((valid >> j) & 1u) {
      const unsigned long long idx = table_find_index(t, c);
      if (idx == ~0ull) {
        atomicAdd(&counters[1], 1ull);
      } else {
        const uint32_t slot = atomicAdd(&cursor[idx], 1u);
        const unsigned long long o = run_off[idx];
        if (o + slot < run_off[idx + 1]) occ[o + slot] = ((p + (uint64_t)j) << 1) | (use_rc ? 1ull : 0ull);
        else atomicAdd(&counters[2], 1ull);
      }
    }
  });
}

// ---------------------------------------------------------------- two-phase build: scatter to buckets, place per bucket
constexpr int OCC_PLACE_NT = 256;
constexpr uint32_t OCC_PLACE_CAP = 2048;   // distinct k-mers of a bucket the shared-memory table holds (24 KB)

// level-1 element of a canonical k-mer: the remainder below the prefix (one-word keys, REM <= 32) or the key
template <typename Elem, int W> struct OccElem;
template <int W> struct OccElem<uint32_t, W> {
  static APGK_HD uint32_t make(const Key<W>& c, int rem_bits, int pad) { return (uint32_t)((c.w[0] << pad) & lowmask64(rem_bits)); }
  static APGK_HD Key<W> key(uint32_t e, uint32_t b, int rem_bits, int pad) {
    Key<W> k;
    k.w[0] = ((rem_bits >= 64 ? 0ull : ((uint64_t)b << rem_bits)) | e) >> pad;
    return k;
  }
};
template <int W> struct OccElem<Key<W>, W> {
  static APGK_HD Key<W> make(const Key<W>& c, int, int) { return c; }
  static APGK_HD Key<W> key(const Key<W>& e, uint32_t, int, int) { return e; }
};

// bstart[b] = first slot of prefix bucket b (b = 0 .. nb); bcur[b] = the bucket's write cursor, starting there
__global__ void k_occ_bstart(const unsigned long long* __restrict__ index, const unsigned long long* __restrict__ run_off,
                             uint32_t nb, unsigned long long* __restrict__ bstart, unsigned long long* __restrict__ bcur) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > nb) return;
  const unsigned long long v = run_off[index[b]];
  bstart[b] = v;
  if (b < nb) bcur[b] = v;
}

// Sweep of the reads: every window takes the next slot of its prefix bucket (ONE 64-bit global atomic on a
// cursor that holds absolute slots: 2^P counters, L2 resident) and stores its element there.  pack_bits > 0
// (32-bit remainders whose REM bits fit above the position in one word): pos_tmp[o] = rem << pack_bits | pos,
// one 8-byte store per window; else the element and the position go to two arrays.  A slot can only run
// past its bucket if the table does not match the read store; k_occ_place would then miss the k-mer.
// Only the windows starting in [first, first + n_bases) take part (the whole store for the single-GPU forms).
// Pos = unsigned long long: pos = (global base position << 1) | canonical-is-reverse; Pos = uint32_t: pos = base
// position - first, never packed (the batches of the group lookups, csrc/gfreq.cuh).  hist != nullptr: the
// sweep only counts the windows of every bucket into hist[b] and places nothing.
template <int W, typename Elem, typename Pos, int NT>
__global__ void __launch_bounds__(NT) k_occ_scatter(ReadStore rs, FreqTable<W> t, uint64_t first, uint64_t n_bases,
                                                    uint32_t* __restrict__ hist, unsigned long long* __restrict__ bcur,
                                                    Elem* __restrict__ elems, Pos* __restrict__ pos_tmp,
                                                    int pack_bits, unsigned long long n_slots,
                                                    unsigned long long* __restrict__ counters) {
  const uint64_t p = (first & ~15ull) + ((uint64_t)blockIdx.x * NT + threadIdx.x) * POS_PER_THREAD;
  const uint64_t end = first + n_bases;
  if (p >= end) return;
  uint32_t valid = window_valid_mask16(rs.starts32, p, rs.K, rs.total_bases);
  if (p < first) valid &= 0xFFFFu << (uint32_t)(first - p);
  if (end - p < 16) valid &= (1u << (uint32_t)(end - p)) - 1u;
  if (!valid) return;
  Window16<W> win;
  load_window16<W>(rs.bases32, p, rs.K, win);
  extract16<W>(win, rs.K, [&](int j, const Key<W>& c, bool use_rc) {
    if ((valid >> j) & 1u) {
      const uint32_t b = digit_of(c, t.prefix_pos, t.prefix_len, t.pad);
      if (hist) { atomicAdd(&hist[b], 1u); return; }
      const unsigned long long o = atomicAdd(&bcur[b], 1ull);   // (a 32-bit relative cursor + a read of bstart[b] measured 10 % slower)
      const unsigned long long pv = ((p + (uint64_t)j) << 1) | (use_rc ? 1ull : 0ull);
      if (o >= n_slots) {
        atomicAdd(&counters[2], 1ull);
      } else if constexpr (sizeof(Pos) == 4) {
        elems[o] = OccElem<Elem, W>::make(c, t.prefix_pos, t.pad);
        pos_tmp[o] = (Pos)(p + (uint64_t)j - first);
      } else if constexpr (sizeof(Elem) == 4) {
        const uint32_t r = OccElem<Elem, W>::make(c, t.prefix_pos, t.pad);
        if (pack_bits) {
          pos_tmp[o] = ((unsigned long long)r << pack_bits) | pv;
        } else {
          elems[o] = r;
          pos_tmp[o] = pv;
        }
      } else {
        elems[o] = OccElem<Elem, W>::make(c, t.prefix_pos, t.pad);
        pos_tmp[o] = pv;
      }
    }
  });
}

// One CTA per prefix bucket.  The CTA walks the bucket's elements NT at a time with a barrier per step,
// so slots are handed out in (nearly) element order and the runs stay almost sorted for the sort pass.
// FREQ = true is the bulk form of the frequency-table lookups error correction makes (apgk_read_freqs over
// the whole store): instead of taking a slot, every element writes its k-mer's count -- the length of
// the run -- to freq_out[its base position]; no atomics, no sort, and the ~10 dependent DRAM accesses of
// a table search per window become one shared-memory search plus one 4-byte store.
template <int W, typename Elem, int NT, bool FREQ>
__global__ void __launch_bounds__(NT) k_occ_place(FreqTable<W> t, const unsigned long long* __restrict__ run_off,
                                                  const unsigned long long* __restrict__ bstart, const Elem* __restrict__ elems,
                                                  const unsigned long long* __restrict__ pos_tmp, int pack_bits,
                                                  uint32_t* __restrict__ cursor, unsigned long long* __restrict__ occ,
                                                  uint32_t* __restrict__ freq_out, unsigned long long* __restrict__ counters) {
  constexpr bool U32 = sizeof(Elem) == 4;
  __shared__ uint32_t sh_rem[U32 ? OCC_PLACE_CAP : 1], sh_off[U32 ? OCC_PLACE_CAP + 1 : 1], sh_cur[U32 ? OCC_PLACE_CAP : 1];
  const unsigned long long pos_mask = pack_bits ? ((1ull << pack_bits) - 1ull) : ~0ull;
  for (uint32_t b = blockIdx.x; b < t.nb; b += gridDim.x) {
    const unsigned long long e0 = bstart[b], n = bstart[b + 1] - e0;
    if (!n) continue;
    const unsigned long long t0 = t.index[b], d = t.index[b + 1] - t0;
    bool in_sh = false;
    if constexpr (U32) in_sh = d <= OCC_PLACE_CAP && n < (1ull << 32);
    if (in_sh) {
      if constexpr (U32) {
        for (uint32_t j = threadIdx.x; j <= (uint32_t)d; j += NT) {
          sh_off[j] = (uint32_t)(run_off[t0 + j] - e0);
          if (j < (uint32_t)d) {
            sh_rem[j] = OccElem<Elem, W>::make(t.keys[t0 + j], t.prefix_pos, t.pad);
            sh_cur[j] = 0;
          }
        }
        __syncthreads();
        for (unsigned long long i0 = 0; i0 < n; i0 += NT) {
          const unsigned long long i = i0 + threadIdx.x;
          unsigned long long pv = 0;
          uint32_t lo = 0xFFFFFFFFu;                 // run of this thread's element (none: past the end / not found)
          if (i < n) {
            pv = pos_tmp[e0 + i];
            uint32_t r;
            if (pack_bits) { r = (uint32_t)(pv >> pack_bits); pv &= pos_mask; } else { r = elems[e0 + i]; }
            uint32_t hi = (uint32_t)d;
            lo = 0;
            while (lo < hi) {
              const uint32_t mid = (lo + hi) >> 1;
              if (sh_rem[mid] < r) lo = mid + 1; else hi = mid;
            }
            if (!(lo < (uint32_t)d && sh_rem[lo] == r)) {
              atomicAdd(&counters[1], 1ull);
              lo = 0xFFFFFFFFu;
            }
          }
          if constexpr (FREQ) {
            if (lo != 0xFFFFFFFFu) freq_out[pv >> 1] = sh_off[lo + 1] - sh_off[lo];
          } else {
            // Slots are handed out warp after warp (a barrier between warps), so a run receives its elements in
            // element order: a k-mer of a 45x genome has 2-3 elements in every 256-element step, and with the
            // warps racing most runs arrived with inversions (the sort pass then took 54 ms instead of ~15).
#pragma unroll 1
            for (int w = 0; w < NT / 32; w++) {
              if ((int)(threadIdx.x >> 5) == w && lo != 0xFFFFFFFFu) {
                const uint32_t slot = sh_off[lo] + atomicAdd(&sh_cur[lo], 1u);
                if (slot < sh_off[lo + 1]) occ[e0 + slot] = pv; else atomicAdd(&counters[2], 1ull);
              }
              __syncthreads();
            }
          }
        }
        if constexpr (FREQ) __syncthreads();       // the shared table is reloaded for the next bucket
      }
    } else {
      for (unsigned long long i0 = 0; i0 < n; i0 += NT) {
        const unsigned long long i = i0 + threadIdx.x;
        if (i < n) {
          unsigned long long pv = pos_tmp[e0 + i];
          Key<W> c;
          if constexpr (U32) {
            uint32_t r;
            if (pack_bits) { r = (uint32_t)(pv >> pack_bits); pv &= pos_mask; } else { r = elems[e0 + i]; }
            c = OccElem<Elem, W>::key(r, b, t.prefix_pos, t.pad);
          } else {
            c = elems[e0 + i];
          }
          const unsigned long long idx = table_find_index(t, c);
          if (idx == ~0ull) {
            atomicAdd(&counters[1], 1ull);
          } else if constexpr (FREQ) {
            freq_out[pv >> 1] = t.counts[idx];
          } else {
            const uint32_t slot = atomicAdd(&cursor[idx], 1u);
            const unsigned long long o = run_off[idx] + slot;
            if (o < run_off[idx + 1]) occ[o] = pv; else atomicAdd(&counters[2], 1ull);
          }
        }
        if constexpr (!FREQ) __syncthreads();
      }
    }
  }
}

// One thread per run.  Insertion sort straight on the run: linear when it arrived sorted.
__global__ void k_occ_sort_small(const unsigned long long* __restrict__ run_off, uint64_t n_runs,
                                 unsigned long long* __restrict__ occ, unsigned long long* __restrict__ big_list,
                                 unsigned long long* __restrict__ counters) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_runs) return;
  const unsigned long long o = run_off[i], n = run_off[i + 1] - o;
  if (n < 2) return;
  if (n > OCC_SMALL_MAX) {
    big_list[atomicAdd(&counters[0], 1ull)] = i;
    return;
  }
  unsigned long long* a = occ + o;
  unsigned long long mx = a[0];  // largest value of the sorted part a[0..j)
  for (uint32_t j = 1; j < (uint32_t)n; j++) {
    const unsigned long long v = a[j];
    if (v < mx) {
      uint32_t k = j;
      while (k > 0 && a[k - 1] > v) { a[k] = a[k - 1]; k--; }
      a[k] = v;
    } else {
      mx = v;
    }
  }
}

// One CTA per big run (grid-stride over the list).  Bitonic network whose every comparison is ascending
// (the first step of a merge compares mirrored partners), so the padding to a power of two can stay
// virtual: a partner at or beyond n counts as +infinity and is never touched.
template <int NT>
__global__ void __launch_bounds__(NT) k_occ_sort_big(const unsigned long long* __restrict__ run_off,
                                                     const unsigned long long* __restrict__ big_list,
                                                     const unsigned long long* __restrict__ counters,
                                                     unsigned long long* __restrict__ occ) {
  __shared__ unsigned long long sh[OCC_SH_CAP];
  const unsigned long long n_big = counters[0];
  for (unsigned long long r = blockIdx.x; r < n_big; r += gridDim.x) {
    const unsigned long long i = big_list[r];
    const unsigned long long o = run_off[i], n = run_off[i + 1] - o;
    unsigned long long* a = occ + o;
    const bool in_sh = n <= OCC_SH_CAP;
    unsigned long long* buf = in_sh ? sh : a;
    if (in_sh) {
      for (unsigned long long j = threadIdx.x; j < n; j += NT) sh[j] = a[j];
    }
    __syncthreads();
    unsigned long long m = 2;
    while (m < n) m <<= 1;
    const unsigned long long half = m >> 1;
    for (unsigned long long k = 2; k <= m; k <<= 1) {
      for (unsigned long long s = k >> 1; s > 0; s >>= 1) {
        const bool mirror = (s == (k >> 1));
        for (unsigned long long t = threadIdx.x; t < half; t += NT) {
          const unsigned long long lo = ((t & ~(s - 1)) << 1) | (t & (s - 1));
          const unsigned long long hi = mirror ? (lo | (k - 1)) - (t & (s - 1)) : lo + s;
          if (hi < n) {
            const unsigned long long x = buf[lo], y = buf[hi];
            if (x > y) { buf[lo] = y; buf[hi] = x; }
          }
        }
        __syncthreads();
      }
    }
    if (in_sh) {
      for (unsigned long long j = threadIdx.x; j < n; j += NT) a[j] = sh[j];
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- global position -> (read id, position in read)
// number of read starts in each block of RANK_BLOCK_WORDS bitmap words
__global__ void k_start_blocks(const uint32_t* __restrict__ starts32, uint64_t n_blocks, uint32_t* __restrict__ cnt) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_blocks) return;
  uint32_t s = 0;
#pragma unroll
  for (int w = 0; w < RANK_BLOCK_WORDS; w++) s += __popc(starts32[i * RANK_BLOCK_WORDS + w]);
  cnt[i] = s;
}

// occ[i] = (q << 1 | rc) -> read_id[i], pos[i]: pos is 1-based in the read, negative when the canonical
// form is the reverse complement of the read's window (SortKmers record convention, SURVEY.md 8(a) [U]).
// Reads without bases own no start bit: empty_nb[e] = non-empty reads before the e-th empty read (ascending)
// shifts the rank back to the caller's read numbering.
__global__ void k_occ_translate(const unsigned long long* __restrict__ occ, uint64_t n, const uint32_t* __restrict__ starts32,
                                const unsigned long long* __restrict__ blk_rank, const unsigned long long* __restrict__ empty_nb,
                                uint32_t n_empty, uint32_t* __restrict__ read_id, int32_t* __restrict__ pos) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long v = occ[i];
  const uint64_t q = v >> 1;
  const uint64_t wq = q >> 5, blk = wq / RANK_BLOCK_WORDS;
  unsigned long long rank = blk_rank[blk];
  for (uint64_t w = blk * RANK_BLOCK_WORDS; w < wq; w++) rank += __popc(starts32[w]);
  uint32_t bits = starts32[wq] & (0xFFFFFFFFu >> (31u - (uint32_t)(q & 31)));  // starts at positions <= q
  rank += __popc(bits);
  uint64_t w = wq;
  while (!bits && w > 0) bits = starts32[--w];
  const uint64_t s = (w << 5) + (bits ? 31u - (uint32_t)__clz((int)bits) : 0u);  // start of the read holding q
  unsigned long long id = rank ? rank - 1 : 0;  // rank among the reads that have bases
  if (n_empty) {
    uint32_t lo = 0, hi = n_empty;               // number of empty reads with empty_nb <= id
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (empty_nb[mid] <= id) lo = mid + 1; else hi = mid;
    }
    id += lo;
  }
  const int32_t p1 = (int32_t)(q - s) + 1;
  read_id[i] = (uint32_t)id;
  pos[i] = (v & 1ull) ? -p1 : p1;
}

}  // namespace apgk
