// local3.cuh -- sort-and-count for 32-bit remainders by ORDER-PRESERVING hashing.
//
// It walks the buckets k_local5 (local5.cuh) defers: those with more distinct keys than k_local5's table or more
// instances than its 16-bit counts.  It takes every bucket size, so it is the fallback.
//
// Keys of one bucket share their leading bits, so the remainder r (< 2^REM) of a
// random-looking genome is spread evenly.  The table is cut into ROWS of 16 slots and
// the row of a key is chosen MONOTONE in the key:   row(r) = floor(r * nrows / 2^REM);
// inside its row a key probes from a scrambled start (multiplicative hash), wrapping
// inside the row.  One CAS + one ADD per key instance groups identical keys.  Rows
// are in ascending key order by construction, so only the <= 16 entries of a row have
// to be ranked against each other: there is no separate sort.
// (Tried and measured no faster, profiles/r01_sweeps.txt "local3 variants": four straight-line first
// probes per thread with the occupancy bitmap rebuilt by one thread per row instead of an atomicOr per
// fresh slot; a two-choice start slot that keeps most warps out of the probing loop; an L2 prefetch of
// the next bucket.  Issue slots and the L1 data pipe both sit at ~60%: the kernel is bound by the
// barrier-separated phases of small buckets, not by instruction count.)
// (Round 2, profiles/r02_local3_experiments.txt: ncu shows 69 % issue-slot utilisation and 2.1 shared atomics per
// key, yet neither a variant with ~40 % fewer instructions on the insert path -- 32-bit shared-window addressing,
// compile-time table offsets, per-pass constants pinned in registers, rolled probe loop, predicate-free full
// batches, branch-free 16-slot row ranking -- nor one that also halved the atomics -- look before CAS, so a
// duplicate costs one RED; no occupancy bitmap -- moved the time (28.0 and 29.8 ms against 28.1).  What does move
// it: the bucket size.  Per-rank timings of the sharded form give t = 4.3 ps x keys + 9.2 ns x buckets per GPU,
// i.e. a bucket costs as much as ~2100 keys whatever it holds (six CTA-wide phases, one exposed global-load
// latency), and larger buckets pay more per key for probing (P = 19: 39 ms).)
// (A fully monotone slot hash was tried first: sequencing-error variants of a genomic
// k-mer differ in their low bits, land on the same home slot and build clusters right
// where the 45x-covered k-mer lives -- ncu showed 6.5 warp instructions per key in
// the probing loop.  The scrambled in-row start removes that.)
//
// A bucket is processed as a stack of DYADIC KEY RANGES (d, i) = "the keys whose
// top d remainder bits equal i", starting with the whole bucket (0, 0).  For one range:
//
//   1. clear table + occupancy bitmap (128-bit stores)                        [block]
//   2. insert the range's keys straight from HBM/L2 (monotone home of the bits
//      below the range prefix); the thread that claims a fresh slot sets its
//      bit in the bitmap                                                      [block]
//   3. bitmap words -> dense list of occupied slots in slot order
//      (popcount + one block scan)                                            [block]
//   4. one thread per DISTINCT key: rank inside its cluster by comparison,
//      write (k-mer, count) at its final ascending position, update the
//      spectrum                                                               [block, all lanes busy]
//
// If a row fills up (too many distinct keys for the table, or a skewed range),
// nothing has been written yet and the range is
// split into its two halves (d+1, 2i), (d+1, 2i+1) -- so oversize and skewed
// buckets take more passes instead of a different kernel.  A range of one key
// value (d == REM) always fits.  (The first version walked table SLOTS in steps
// 3-4: ncu showed 10 warp instructions per key with ~3 of 32 lanes active.)
#pragma once
#include "local2.cuh"

#ifndef L3_PREFETCH
#define L3_PREFETCH 1
#endif
namespace apgk {

constexpr int L3_ROW = 16;      // slots per row (a row is half a bitmap word)
constexpr int L3_SLACK = 96;    // table padding
constexpr int L3_STACK = 72;    // >= 2 * 32 pending ranges

// Needs 1 <= REM <= 31.  Shared memory (NS = slots(LM)):
//   key[NS] u32 | cnt[NS] u32 | bitmap[NS/32] u32 | spec[SPEC_SMEM] | wsum[40] | misc[8] | stack[2*L3_STACK] | list[LM] u16
struct Local3Smem {
  uint32_t* key; uint32_t* cnt; uint32_t* bitmap; uint16_t* list; uint32_t* spec; uint32_t* wsum; uint32_t* misc;
  uint32_t* stack;
  static __host__ __device__ size_t slots(int LM) { return (((size_t)LM + LM / 4 + 1 + L3_SLACK) + 127) & ~(size_t)127; }
  __device__ __forceinline__ void carve(unsigned char* raw, int LM) {
    const size_t ns = slots(LM);
    key = (uint32_t*)raw;
    cnt = key + ns;
    bitmap = cnt + ns;
    spec = bitmap + ns / 32 + 4;
    wsum = spec + SPEC_SMEM;
    misc = wsum + 40;
    stack = misc + 8;
    list = (uint16_t*)(stack + 2 * L3_STACK);
  }
  static size_t bytes(int LM) {
    return (slots(LM) * 2 + slots(LM) / 32 + 4 + SPEC_SMEM + 40 + 8 + 2 * L3_STACK) * 4 + ((size_t)LM + LM / 4 + 128) * 2 + 16;
  }
};

// Buckets list[1 .. 1 + min(list[0], list_cap)).
template <int NT, int W>
__global__ void __launch_bounds__(NT, 1536 / NT) k_local3(const uint32_t* __restrict__ src, BucketTable bt, int rem_bits, EmitCtx<W> ec,
                                               uint32_t* __restrict__ nd_out, const uint32_t* __restrict__ list,
                                               uint32_t list_cap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Local3Smem sm;
  const int LM = (int)bt.local_max;
  sm.carve(smem_raw, LM);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  constexpr int NWARP = NT / 32;
  for (int i = tid; i < SPEC_SMEM; i += NT) sm.spec[i] = 0;
  const int up = 32 - rem_bits;                       // remainder left-aligned in 32 bits
  const uint32_t m_cap = (uint32_t)LM + (uint32_t)LM / 4 + 1;  // homes of a full-size pass
  // The next bucket's size / offset are loaded one bucket ahead and its keys are pulled toward L2 while
  // the current bucket is processed: a CTA otherwise sits through two dependent DRAM latencies per
  // bucket (bsize/bofs, then the keys) and three CTAs per SM do not cover them.
  const uint32_t n_iter = list[0] < list_cap ? list[0] : list_cap;
  uint32_t b_nx = 0;
  unsigned long long n_nx = 0, o_nx = 0;
  if (blockIdx.x < n_iter) { b_nx = list[1 + blockIdx.x]; n_nx = bt.bsize[b_nx]; o_nx = bt.bofs[b_nx]; }
  for (uint32_t it = blockIdx.x; it < n_iter; it += gridDim.x) {
    const uint32_t b = b_nx;
    const unsigned long long n64 = n_nx;
    const unsigned long long o = o_nx;
    {
      const uint32_t itn = it + gridDim.x;
      if (itn < n_iter) { b_nx = list[1 + itn]; n_nx = bt.bsize[b_nx]; o_nx = bt.bofs[b_nx]; }
    }
    if (n64 == 0) {
      if (tid == 0) nd_out[b] = 0;
      continue;
    }
    const uint32_t* s = src + o;
    // a pass over a small bucket only needs a small table
    const uint32_t m_want = n64 < (unsigned long long)LM ? (uint32_t)n64 + ((uint32_t)n64 >> 2) + 1 : m_cap;
    const uint32_t nrows = (m_want + L3_ROW - 1) / L3_ROW;
    const uint32_t ns = nrows * L3_ROW;                // slots in use
    const uint32_t ns4 = (ns + 3) >> 2;                // uint4 groups to clear (table is padded to 128 slots)
    const uint32_t nwords = (ns + 31) >> 5;
    volatile uint32_t* vmisc = sm.misc;
    uint32_t run_nd = 0;                               // records already emitted for this bucket
    bool first = true;                                 // the first range is the whole bucket: (d=0, i=0)
    while (true) {
      __syncthreads();  // previous pass / previous bucket fully emitted (table, stack and misc are reused)
      uint32_t sp = 1, rd = 0, ri = 0;
      if (!first) {
        sp = sm.misc[1];
        if (sp == 0) break;
        rd = sm.stack[2 * (sp - 1)];
        ri = sm.stack[2 * (sp - 1) + 1];
      }
      first = false;
      // ---- 1. clear
      {
        uint4* k4 = reinterpret_cast<uint4*>(sm.key);
        uint4* c4 = reinterpret_cast<uint4*>(sm.cnt);
        const uint4 e4 = make_uint4(SLOT_EMPTY, SLOT_EMPTY, SLOT_EMPTY, SLOT_EMPTY), z4 = make_uint4(0, 0, 0, 0);
        for (uint32_t i = tid; i < ns4; i += NT) { k4[i] = e4; c4[i] = z4; }
        for (uint32_t i = tid; i < nwords + 2; i += NT) sm.bitmap[i] = 0;
        if (tid == 0) sm.misc[0] = 0;   // "this pass failed" flag; nobody touches it between the two barriers
      }
      __syncthreads();
      if (tid == 0) sm.misc[1] = sp - 1;  // pop (every thread has read sp and the range before the barrier)
      // ---- 2. insert the keys of range (rd, ri); 4 independent loads in flight per thread
      const uint32_t pshift = 32 - rd;                 // x >> pshift = top rd bits (rd == 0: everything matches)
      for (unsigned long long i0 = 0; i0 < n64; i0 += 4ull * NT) {
        uint32_t kk[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned long long i = i0 + (unsigned long long)u * NT + tid;
          kk[u] = i < n64 ? s[i] : SLOT_EMPTY;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const uint32_t k = kk[u];
          const uint32_t x = k << up;
          // in range?  (k == EMPTY marks the tail of the bucket; remainders are < 2^31)
          if (k != SLOT_EMPTY && (rd == 0 || (x >> pshift) == ri)) {
            const uint32_t row = __umulhi(x << rd, nrows) * L3_ROW;  // monotone in the bits below the range prefix
            uint32_t h = (k * 0x9E3779B1u) >> 28;                    // scrambled start inside the row
            // first probe, branch-light: one unconditional CAS answers "empty, mine, or someone else's"
            uint32_t slot = row + h;
            uint32_t cur = atomicCAS(&sm.key[slot], SLOT_EMPTY, k);
            if (cur == SLOT_EMPTY) atomicOr(&sm.bitmap[slot >> 5], 1u << (slot & 31));
            bool placed = (cur == SLOT_EMPTY) | (cur == k);
            for (int pr = 1; !placed; pr++) {          // a few % of the keys: probe on, wrapping inside the row
              if (pr == L3_ROW) { sm.misc[0] = 1u; break; }          // row full: this range needs splitting
              h = (h + 1) & (L3_ROW - 1);
              slot = row + h;
              cur = atomicCAS(&sm.key[slot], SLOT_EMPTY, k);
              if (cur == SLOT_EMPTY) atomicOr(&sm.bitmap[slot >> 5], 1u << (slot & 31));
              placed = (cur == SLOT_EMPTY) | (cur == k);
            }
            if (placed) atomicAdd(&sm.cnt[slot], 1u);
          }
          // Reconverge the warp after every key: without this the lanes that finish probing early run
          // ahead on their own (independent thread scheduling) and the whole loop executes with ~14 of
          // 32 lanes active (ncu: LDG of the next batch issued 3x more often than needed).
          __syncwarp();
        }
        if (n64 > (unsigned long long)LM && __any_sync(0xffffffffu, vmisc[0] != 0)) break;  // failed pass of a big bucket
      }
      __syncthreads();
#if L3_PREFETCH
      if (L3_PREFETCH == 1 || run_nd == 0) {  // next bucket's keys toward L2 (32 keys per 128-byte line)
        const unsigned long long i = (unsigned long long)tid * 32;
        if (it + gridDim.x < n_iter && i < n_nx && tid < 1024) prefetch_l2(src + o_nx + i);
      }
#endif
      // ---- 3. dense list of occupied slots, in slot order
      uint32_t nd_total;
      {
        constexpr int WPT = 2;  // bitmap words per thread; nwords <= NT * WPT (host: LM vs NT)
        uint32_t wd[WPT], c = 0;
#pragma unroll
        for (int u = 0; u < WPT; u++) {
          const uint32_t wi = tid * WPT + u;
          wd[u] = wi < nwords ? sm.bitmap[wi] : 0u;
          c += __popc(wd[u]);
        }
        const uint32_t incl = warp_incl_scan(c, lane);
        if (lane == 31) sm.wsum[wid] = incl;
        __syncthreads();
        uint32_t base = incl - c;
        nd_total = 0;
#pragma unroll
        for (int w = 0; w < NWARP; w++) {
          const uint32_t v = sm.wsum[w];
          if (w < wid) base += v;
          nd_total += v;
        }
        const bool failed = sm.misc[0] != 0;
        if (!failed) {
#pragma unroll
          for (int u = 0; u < WPT; u++) {
            uint32_t w = wd[u];
            const uint32_t s_base = (tid * WPT + u) << 5;
            while (w) {
              const int bit = __ffs((int)w) - 1;
              w &= w - 1;
              sm.list[base++] = (uint16_t)(s_base + bit);
            }
          }
        }
      }
      __syncthreads();
      if (sm.misc[0] != 0) {
        // nothing was written or counted: split the range (a one-value range cannot fail)
        if (tid == 0) {
          uint32_t top = sm.misc[1];
          if ((int)rd < rem_bits && top + 2 <= L3_STACK) {
            sm.stack[2 * top] = rd + 1; sm.stack[2 * top + 1] = 2 * ri + 1; top++;   // upper half, popped second
            sm.stack[2 * top] = rd + 1; sm.stack[2 * top + 1] = 2 * ri; top++;       // lower half, popped first
            sm.misc[1] = top;
          } else {
            sm.misc[2] = 1u;  // cannot happen for valid input; surfaces as a count mismatch rather than a hang
          }
        }
        continue;
      }
      // ---- 4. one thread per distinct key: rank inside the cluster, emit
      for (uint32_t j0 = 0; j0 < nd_total; j0 += NT) {
        const uint32_t j = j0 + tid;
        uint32_t f = 0;
        if (j < nd_total) {
          const uint32_t q = sm.list[j];
          const uint32_t k = sm.key[q];
          // the row's occupancy is one half of a bitmap word; rank k among the row's keys
          const uint32_t rbase = q & ~(uint32_t)(L3_ROW - 1);
          uint32_t rowbits = (sm.bitmap[q >> 5] >> (rbase & 31)) & 0xFFFFu;
          const uint32_t before = __popc(rowbits & ((1u << (q & (L3_ROW - 1))) - 1u));
          uint32_t smaller = 0;
          while (rowbits) {
            const int bit = __ffs((int)rowbits) - 1;
            rowbits &= rowbits - 1;
            smaller += sm.key[rbase + bit] < k;
          }
          const unsigned long long pos = o + run_nd + (j - before + smaller);
          f = sm.cnt[q];
          if (ec.want_table) {
            ec.tmp_keys[pos] = rebuild_key<W>(k, (uint64_t)b, ec.rem_bits, ec.pad);
            ec.tmp_cnt[pos] = f;
          }
        }
        // spectrum: singletons dominate, so they are counted per warp with one ballot
        const uint32_t ones = __ballot_sync(0xffffffffu, f == 1u);
        if (lane == 0 && ones) atomicAdd(&sm.spec[1], (uint32_t)__popc(ones));
        if (f > 1u) {
          if (f < SPEC_SMEM) atomicAdd(&sm.spec[f], 1u);
          else spec_add_global(ec.spec_dense, ec.spec_ovf, ec.spec_ovf_cap, f);
        }
      }
      run_nd += nd_total;
      if (sm.misc[1] == 0) break;  // stack empty (written by thread 0 before the last barriers): bucket done
    }
    if (tid == 0) nd_out[b] = run_nd;
  }
  __syncthreads();
  for (int i = tid; i < SPEC_SMEM; i += NT) {
    const uint32_t v = sm.spec[i];
    if (v) atomicAdd(&ec.spec_dense[i], (unsigned long long)v);
  }
}

}  // namespace apgk
