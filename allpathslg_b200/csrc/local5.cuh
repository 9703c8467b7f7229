// local5.cuh -- sort-and-count for 32-bit remainders: a SMALL CTA per bucket with a table sized by DISTINCT keys.
//
// k_local3 gives every bucket a 512-thread CTA whose table is sized by instances (~5.4 k slots at the bench
// geometry, ~11 % full) and runs three CTAs per SM.  Here a 128-thread CTA owns one bucket at a time with a
// 2048-slot table, so eight CTAs share an SM and their barriers overlap each other:
//
//   1. insert: 16-byte loads, the next batch in flight while the current one is inserted; one CAS + one RED per
//      instance (linear probing from a scrambled start over the whole table, a __syncwarp after every key so the
//      lanes that probe further do not split the warp); a fresh slot sets its bit in the occupancy bitmap and
//      counts one key for its GROUP, the top L5_GBITS bits of the remainder
//   2. one warp scan of the group counts; the occupied slots are scattered into a list grouped by group (a
//      counting sort: groups ascend in key order)
//   3. one thread per distinct key: rank inside its group by comparison, write (k-mer, count) at its final
//      ascending position, update the spectrum
//   4. clear the table for the next bucket (128-bit stores)
//
// Why not k_local3's rows (a row chosen monotone in the key, so rows need no sort) in a small table?  Keys cluster
// in key space: sequencing-error variants and the genome's repeats share a k-mer's leading bases.  At 2048 slots,
// rows of 32 chosen by the top remainder bits overflow in 28 % of the buckets of the bench's reads
// (tools/local_table_sim.py, profiles/r04_local_warp.txt).  A hash over the whole table does not see the clusters;
// they only make some groups larger, which costs comparisons (6.2 per key on average with 8 group bits).
//
// Table size.  A bucket holds ~590 distinct keys on average at the bench geometry (2^20 buckets, 617 M distinct
// k-mers), ~1250 at the 99th percentile and ~1420 at most (the densest canonical prefixes).  2048 slots take up to
// L5_DMAX = 1536 (75 % load).  Counts are 16 bits, two to a word, which the instance cap L5_NMAX makes safe.
// A CTA's shared memory is 8 KB keys + 4 KB counts + 2 KB group counts and cursors + 256 B bitmap + 3 KB list +
// 1 KB spectrum = 18.4 KB; eight CTAs (32 warps) per SM need <= 64 registers per thread (ptxas: 52, no spills).
// Measured on the bench (local stage, ms): 128 threads 24.7, 256 threads 25.9, 512 threads 35.9; 128 threads with
// 11 CTAs per SM forced (40 registers, spills) 24.4 -- not worth the spills (profiles/r04_local_warp.txt).
// (One WARP per bucket with the same table, 12 warps per SM, was 2.4x slower than k_local3: the insert is bound by
// latency and shared atomics, and needs many warps per SM -- profiles/r04_local_warp.txt.)
//
// A bucket goes on the deferred list -- nothing is written for it, k_local3 takes it afterwards -- when it holds
// more than L5_NMAX instances or more than L5_DMAX distinct keys.
#pragma once
#include "local2.cuh"

namespace apgk {

constexpr int L5_NT = 128;                            // threads per CTA (one bucket at a time)
constexpr int L5_NW = L5_NT / 32;
constexpr int L5_SLOTS = 2048;
constexpr int L5_SLOT_BITS = 11;
constexpr uint32_t L5_DMAX = 1536;                    // distinct keys per bucket (75 % load)
constexpr uint32_t L5_NMAX = 65535;                   // instances per bucket (16-bit counts)
constexpr int L5_GBITS = 8;                           // group = top 8 remainder bits
constexpr int L5_GROUPS = 1 << L5_GBITS;
constexpr int L5_SPEC = 256;                          // shared spectrum bins (larger counts: global atomics)
constexpr int L5_U = 2;                               // 16-byte loads per thread and batch
// spec[L5_SPEC] | wsum[2][L5_NW] (32 words) | key[SLOTS] | cnt[SLOTS/2] | gcnt[GROUPS] | gcur[GROUPS] | bitmap[SLOTS/32] | list[DMAX] u16
constexpr size_t L5_SMEM = (size_t)L5_SPEC * 4 + 128 + (size_t)L5_SLOTS * 4 + (size_t)L5_SLOTS * 2 + (size_t)L5_GROUPS * 8 +
                           L5_SLOTS / 8 + (size_t)L5_DMAX * 2;

template <int W>
__global__ void __launch_bounds__(L5_NT, 8) k_local5(const uint32_t* __restrict__ src, BucketTable bt, int rem_bits,
                                                     EmitCtx<W> ec, uint32_t* __restrict__ nd_out,
                                                     uint32_t* __restrict__ deferred, uint32_t deferred_cap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  uint32_t* spec = reinterpret_cast<uint32_t*>(smem_raw);
  uint32_t* wsum = spec + L5_SPEC;                    // [2][L5_NW] claims per warp, alternating per batch
  uint32_t* key = wsum + 32;
  uint32_t* cnt = key + L5_SLOTS;
  uint32_t* gcnt = cnt + L5_SLOTS / 2;
  uint32_t* gcur = gcnt + L5_GROUPS;
  uint32_t* bitmap = gcur + L5_GROUPS;
  uint16_t* list = reinterpret_cast<uint16_t*>(bitmap + L5_SLOTS / 32);
  // key, cnt, gcnt (contiguous) and bitmap are cleared with 128-bit stores; gcur is rewritten per bucket
  auto clear = [&]() {
    const uint4 e4 = make_uint4(SLOT_EMPTY, SLOT_EMPTY, SLOT_EMPTY, SLOT_EMPTY), z4 = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < L5_SLOTS / 4; i += L5_NT) reinterpret_cast<uint4*>(key)[i] = e4;
    for (int i = tid; i < (L5_SLOTS / 2 + L5_GROUPS) / 4; i += L5_NT) reinterpret_cast<uint4*>(cnt)[i] = z4;
    if (tid < L5_SLOTS / 128) reinterpret_cast<uint4*>(bitmap)[tid] = z4;
  };
  for (int i = tid; i < L5_SPEC; i += L5_NT) spec[i] = 0;
  clear();
  const int up = 32 - rem_bits;                       // remainder left-aligned in 32 bits
  // one key: returns 1 if it claimed a fresh slot, 0 if it found its key, 2 if the table is full
  auto insert = [&](uint32_t k) -> uint32_t {
    uint32_t r = 0;
    if (k != SLOT_EMPTY) {
      uint32_t s = (k * 0x9E3779B1u) >> (32 - L5_SLOT_BITS);   // scrambled start slot
      uint32_t x = atomicCAS(&key[s], SLOT_EMPTY, k);
      for (int pr = 1; x != SLOT_EMPTY && x != k; pr++) {
        if (pr == L5_SLOTS) { r = 2; break; }
        s = (s + 1) & (L5_SLOTS - 1);
        x = atomicCAS(&key[s], SLOT_EMPTY, k);
      }
      if (x == SLOT_EMPTY) {
        atomicOr(&bitmap[s >> 5], 1u << (s & 31));
        atomicAdd(&gcnt[(k << up) >> (32 - L5_GBITS)], 1u);
        r = 1;
      }
      if (r != 2) atomicAdd(&cnt[s >> 1], 1u << ((s & 1) << 4));
    }
    // reconverge after every key: lanes that probed further would otherwise run the rest of the batch apart
    __syncwarp();
    return r;
  };
  uint32_t b = bt.b0 + blockIdx.x;
  unsigned long long n_nx = 0, o_nx = 0;              // the next bucket's size and offset, loaded one bucket ahead
  if (b < bt.nb) { n_nx = bt.bsize[b]; o_nx = bt.bofs[b]; }
  for (; b < bt.nb; b += gridDim.x) {
    const unsigned long long n64 = n_nx, o = o_nx;
    if (b + gridDim.x < bt.nb) { n_nx = bt.bsize[b + gridDim.x]; o_nx = bt.bofs[b + gridDim.x]; }
    if (n64 == 0) {
      if (tid == 0) nd_out[b] = 0;
      continue;
    }
    if (n64 > L5_NMAX) {                              // the table is still clear
      if (tid == 0) {
        const uint32_t i = atomicAdd(&deferred[0], 1u);
        if (i < deferred_cap) deferred[1 + i] = b;
      }
      continue;
    }
    __syncthreads();                                  // the previous bucket's clear is done
    const uint32_t n = (uint32_t)n64;
    // ---- 1. insert.  Elements before the first 16-byte boundary (head) and after the last one (tail) are loaded
    //      singly by threads 0-3 / 4-7; the whole vectors in between 4 to a thread.
    const uint32_t head = (uint32_t)min((unsigned long long)((4u - (uint32_t)(o & 3)) & 3u), n64);
    const uint32_t nv = (n - head) >> 2;
    const uint32_t tail0 = head + 4 * nv;
    uint32_t claimed = 0;
    {
      uint32_t k1 = SLOT_EMPTY;
      if (tid < 4) { if ((uint32_t)tid < head) k1 = src[o + tid]; }
      else if (tid < 8) { if (tail0 + (uint32_t)(tid - 4) < n) k1 = src[o + tail0 + (tid - 4)]; }
      const uint32_t r = insert(k1);
      claimed = r == 2 ? 0x10000u : r;
    }
    const uint4* v = reinterpret_cast<const uint4*>(src + o + head);
    constexpr uint32_t BATCH = L5_NT * L5_U;
    const uint4 empty4 = make_uint4(SLOT_EMPTY, SLOT_EMPTY, SLOT_EMPTY, SLOT_EMPTY);
    uint4 cur[L5_U];
#pragma unroll
    for (int u = 0; u < L5_U; u++) {
      const uint32_t vi = (uint32_t)u * L5_NT + tid;
      cur[u] = vi < nv ? __ldg(v + vi) : empty4;
    }
    // claimed: fresh slots of this thread, + 0x10000 once it found the table full; after every batch the CTA's
    // total decides whether the bucket can stay (uniform: every thread reads the same batch's partial sums)
    uint32_t total = 0;
    for (uint32_t v0 = 0, it = 0;; v0 += BATCH, it++) {
      if (v0 < nv) {
        uint4 nxt[L5_U];
#pragma unroll
        for (int u = 0; u < L5_U; u++) {
          const uint32_t vi = v0 + BATCH + (uint32_t)u * L5_NT + tid;
          nxt[u] = vi < nv ? __ldg(v + vi) : empty4;
        }
#pragma unroll
        for (int u = 0; u < L5_U; u++) {
          const uint32_t kk[4] = {cur[u].x, cur[u].y, cur[u].z, cur[u].w};
#pragma unroll
          for (int c = 0; c < 4; c++) {
            const uint32_t r = insert(kk[c]);
            claimed += r == 2 ? 0x10000u : r;
          }
        }
#pragma unroll
        for (int u = 0; u < L5_U; u++) cur[u] = nxt[u];
      }
      const uint32_t ws = __reduce_add_sync(0xffffffffu, claimed);
      if (lane == 0) wsum[(it & 1) * L5_NW + wid] = ws;
      __syncthreads();
      total = 0;
#pragma unroll
      for (int w = 0; w < L5_NW; w++) total += wsum[(it & 1) * L5_NW + w];
      if (v0 + BATCH >= nv || total > L5_DMAX) break;
    }
    if (total > L5_DMAX) {
      // too many distinct keys (or a full table): nothing was written; k_local3 splits the bucket's key range
      if (tid == 0) {
        const uint32_t i = atomicAdd(&deferred[0], 1u);
        if (i < deferred_cap) deferred[1 + i] = b;
      }
      __syncthreads();
      clear();
      continue;
    }
    const uint32_t nd = total;
    // ---- 2. counting sort of the occupied slots by group: group starts (warp 0, 8 consecutive groups a lane) ...
    if (wid == 0) {
      constexpr int GPL = L5_GROUPS / 32;
      uint32_t gc[GPL], sum = 0;
#pragma unroll
      for (int i = 0; i < GPL; i++) { gc[i] = gcnt[lane * GPL + i]; sum += gc[i]; }
      uint32_t run = warp_incl_scan(sum, lane) - sum;
#pragma unroll
      for (int i = 0; i < GPL; i++) { gcur[lane * GPL + i] = run; run += gc[i]; }
    }
    __syncthreads();
    // ... then the occupied slots of each bitmap word go to their group's cursor
    for (int wi = tid; wi < L5_SLOTS / 32; wi += L5_NT) {
      for (uint32_t w = bitmap[wi]; w; w &= w - 1) {
        const uint32_t s = (uint32_t)wi * 32 + __ffs((int)w) - 1;
        const uint32_t pos = atomicAdd(&gcur[(key[s] << up) >> (32 - L5_GBITS)], 1u);
        list[pos] = (uint16_t)s;
      }
    }
    __syncthreads();
    // ---- 3. one thread per distinct key: rank inside its group, emit
    for (uint32_t j0 = 0; j0 < nd; j0 += L5_NT) {
      const uint32_t j = j0 + tid;
      uint32_t f = 0;
      if (j < nd) {
        const uint32_t q = list[j];
        const uint32_t k = key[q];
        const uint32_t g = (k << up) >> (32 - L5_GBITS);
        const uint32_t ge = gcur[g], gs = ge - gcnt[g];
        uint32_t smaller = 0;
        for (uint32_t i = gs; i < ge; i++) smaller += key[list[i]] < k;
        const unsigned long long pos = o + gs + smaller;
        f = (cnt[q >> 1] >> ((q & 1) << 4)) & 0xFFFFu;
        if (ec.want_table) {
          ec.tmp_keys[pos] = rebuild_key<W>(k, (uint64_t)b, ec.rem_bits, ec.pad);
          ec.tmp_cnt[pos] = f;
        }
      }
      // spectrum: singletons dominate, so they are counted per warp with one ballot
      const uint32_t ones = __ballot_sync(0xffffffffu, f == 1u);
      if (lane == 0 && ones) atomicAdd(&spec[1], (uint32_t)__popc(ones));
      if (f > 1u) {
        if (f < L5_SPEC) atomicAdd(&spec[f], 1u);
        else spec_add_global(ec.spec_dense, ec.spec_ovf, ec.spec_ovf_cap, f);
      }
    }
    if (tid == 0) nd_out[b] = nd;
    // ---- 4. clear for the next bucket
    __syncthreads();
    clear();
  }
  __syncthreads();
  for (int i = tid; i < L5_SPEC; i += L5_NT) {
    const uint32_t x = spec[i];
    if (x) atomicAdd(&ec.spec_dense[i], (unsigned long long)x);
  }
}

}  // namespace apgk
