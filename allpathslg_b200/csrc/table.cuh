// table.cuh -- the k-mer frequency table: compaction of per-bucket records into
// one sorted (k-mer, count) table with a prefix index, and the lookups error
// correction makes against it ("k-mer frequency tables consumed by FindErrors",
// BASELINE.json north_star; SURVEY.md section 3.2 -- no file:line available).
#pragma once
#include "local4.cuh"
#include "local5.cuh"

namespace apgk {

// ---------------------------------------------------------------- exclusive scan of u32 -> u64 (three kernels)
constexpr int SCAN_NT = 1024;
constexpr int SCAN_ITEMS = 4;
constexpr int SCAN_BLOCK = SCAN_NT * SCAN_ITEMS;

__global__ void __launch_bounds__(SCAN_NT) k_scan_blocksum(const uint32_t* __restrict__ in, uint64_t n,
                                                           unsigned long long* __restrict__ blocksum) {
  __shared__ uint32_t scratch[34];
  const uint64_t base = (uint64_t)blockIdx.x * SCAN_BLOCK + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; j++) if (base + j < n) s += in[base + j];
  block_excl_scan<SCAN_NT>(s, scratch);
  if (threadIdx.x == 0) blocksum[blockIdx.x] = scratch[32];
}
// single block: exclusive scan of blocksum[nblocks] in place; total -> blocksum[nblocks]
__global__ void __launch_bounds__(SCAN_NT) k_scan_top(unsigned long long* blocksum, uint32_t nblocks,
                                                      unsigned long long* __restrict__ total_out /* may be null */) {
  __shared__ unsigned long long part[SCAN_NT];
  const uint32_t per = (nblocks + SCAN_NT - 1) / SCAN_NT;
  const uint32_t b0 = threadIdx.x * per;
  unsigned long long s = 0;
  for (uint32_t j = 0; j < per; j++) if (b0 + j < nblocks) s += blocksum[b0 + j];
  part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long run = 0;
    for (int i = 0; i < SCAN_NT; i++) { unsigned long long v = part[i]; part[i] = run; run += v; }
    blocksum[nblocks] = run;
    if (total_out) *total_out = run;
  }
  __syncthreads();
  unsigned long long run = part[threadIdx.x];
  for (uint32_t j = 0; j < per; j++) {
    if (b0 + j < nblocks) { unsigned long long v = blocksum[b0 + j]; blocksum[b0 + j] = run; run += v; }
  }
}
__global__ void __launch_bounds__(SCAN_NT) k_scan_apply(const uint32_t* __restrict__ in, uint64_t n,
                                                        const unsigned long long* __restrict__ blocksum,
                                                        unsigned long long* __restrict__ out /* [n+1] */) {
  __shared__ uint32_t scratch[34];
  const uint64_t base = (uint64_t)blockIdx.x * SCAN_BLOCK + (uint64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; j++) { v[j] = base + j < n ? in[base + j] : 0u; s += v[j]; }
  unsigned long long run = blocksum[blockIdx.x] + block_excl_scan<SCAN_NT>(s, scratch);
#pragma unroll
  for (int j = 0; j < SCAN_ITEMS; j++) {
    if (base + j < n) out[base + j] = run;
    run += v[j];
  }
  if (base <= n && n < base + SCAN_ITEMS) out[n] = run;  // the thread owning index n writes the total
}

// ---------------------------------------------------------------- classify level-1 buckets
// big_list <- ids of buckets larger than local_max; stats[0] = how many, stats[1] = their total size.
__global__ void k_classify(const unsigned long long* __restrict__ bsize, uint32_t nb, uint32_t local_max,
                           uint32_t* __restrict__ big_list, uint32_t big_cap, unsigned long long* __restrict__ stats) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const unsigned long long n = bsize[b];
  if (n > local_max) {
    unsigned long long i = atomicAdd(&stats[0], 1ull);
    atomicAdd(&stats[1], n);
    if (i < big_cap) big_list[i] = b;
  }
}

// ---------------------------------------------------------------- sharded counting: pieces -> buckets
// After the exchange a rank holds, for every bucket b it owns (lo <= b < hi), one piece from each source
// rank s (sizes_all[s][b] elements), laid out source-major.  These kernels merge the sizes and gather the
// pieces into one bucket-major array, so the per-bucket kernels run unchanged on the shard.
__global__ void k_merge_sizes(const uint32_t* __restrict__ sizes_all, uint32_t n_src, uint32_t nb, uint32_t lo, uint32_t hi,
                              uint32_t* __restrict__ bsize32, unsigned int* __restrict__ overflow) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  unsigned long long t = 0;
  if (b >= lo && b < hi)
    for (uint32_t s = 0; s < n_src; s++) t += sizes_all[(size_t)s * nb + b];
  if (t >= (1ull << 32)) { atomicExch(overflow, 1u); t = 0; }
  bsize32[b] = (uint32_t)t;
}
__global__ void k_mask_sizes(const uint32_t* __restrict__ sizes, uint32_t nb, uint32_t lo, uint32_t hi, uint32_t* __restrict__ out) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nb) out[b] = (b >= lo && b < hi) ? sizes[b] : 0u;
}

// split digit of a level-1 element: bits [pos, pos+len) of the remainder (32-bit elements) or of the key
__device__ __forceinline__ uint32_t split_digit(uint32_t e, int pos, uint32_t mask) { return (e >> pos) & mask; }
template <int W>
__device__ __forceinline__ uint32_t split_digit(const Key<W>& e, int pos, uint32_t mask) { return mask ? key_bits(e, pos, __popc(mask)) : 0u; }
__device__ __forceinline__ uint32_t split_strip(uint32_t e, int pos) { return e & lowmask32(pos); }  // keep the bits below the digit
template <int W>
__device__ __forceinline__ Key<W> split_strip(const Key<W>& e, int) { return e; }

// Sender side: sizes of the 2^d2 sub-buckets of every bucket of this rank's partition buffer
// (sub[(b << d2) | j]), so that the receivers can place the pieces in ONE pass over NVLink.
// One WARP per bucket (no barriers, eight buckets in flight per CTA); lane j accumulates bin j.
template <typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_sub_hist(const Elem* __restrict__ elems, const unsigned long long* __restrict__ bofs,
                                                 const unsigned long long* __restrict__ bsize, uint32_t nb, int d2, int digit_pos,
                                                 uint32_t* __restrict__ sub) {
  constexpr int U = 8;
  const uint32_t nbins = 1u << d2, mask = nbins - 1u;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * NT + threadIdx.x) >> 5, nwarps = (gridDim.x * NT) >> 5;
  for (uint32_t b = warp; b < nb; b += nwarps) {
    const uint32_t n = (uint32_t)bsize[b];
    const Elem* src = elems + bofs[b];
    uint32_t mine = 0;
    for (uint32_t i0 = 0; i0 < n; i0 += 32 * U) {
      uint32_t d[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const uint32_t i = i0 + u * 32 + lane;
        d[u] = i < n ? split_digit(src[i], digit_pos, mask) : 0xFFFFFFFFu;
      }
      for (uint32_t j = 0; j < nbins; j++) {
        uint32_t cnt = 0;
#pragma unroll
        for (int u = 0; u < U; u++) cnt += __popc(__ballot_sync(0xffffffffu, d[u] == j));
        if (lane == j) mine += cnt;
      }
    }
    if (lane < nbins) sub[((size_t)b << d2) | lane] = mine;
  }
}

// What the gather reads and writes.  Source s's pieces start at src_base[s] + seg_off[s]: either segments of
// one receive buffer (after an NCCL all-to-all) or the senders' own partition buffers mapped over NVLink peer
// memory -- then the kernel IS the exchange, the loads cross NVLink and no receive buffer exists.
template <typename Elem>
struct GatherArgs {
  const Elem* const* src_base;            // [n_src] base of every source's elements
  const unsigned long long* seg_off;      // [n_src] element offset added to src_base[s] (null: 0)
  const unsigned long long* piece_off;    // [n_src][nb + 1] offset of bucket b's piece in source s
  const uint32_t* sizes_all;              // [n_src][nb] piece sizes
  const unsigned long long* bofs_coarse;  // [nb] offset of merged bucket b in the shard, plus coarse_base
  unsigned long long coarse_base;
  uint32_t n_src, nb, lo, hi;             // owned buckets [lo, hi)
  int d2, digit_pos;                      // split every merged bucket by the d2 bits at digit_pos
  Elem* out;                              // the bucket-major shard
  unsigned long long* bsize_fine;         // [nb << d2] sizes / offsets of the fine buckets (b << d2) | j
  unsigned long long* bofs_fine;
  const uint32_t* sub_sizes;              // [n_src][(hi - lo) << d2] senders' sub-bucket counts of this range, or null
  const uint32_t* const* sub_ptrs;        // [n_src] the senders' own full count arrays [nb << d2] (peer memory), or null
};

// One WARP per owned bucket (grid-stride).  A merged bucket holds n_src times the instances the sender's
// geometry aimed at, so the gather also SPLITS it by the next d2 remainder bits into 2^d2 sub-buckets.
// With the senders' sub-bucket counts at hand the pieces are read ONCE (peer memory is not cached in the
// reader's L2); without them a first pass over the pieces counts.  Order inside a sub-bucket is arbitrary --
// the counting kernels do not depend on it.  Writes the fine bucket table (sizes, offsets).
template <typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_gather_split(const GatherArgs<Elem> ga) {
  // lane j keeps the count and then the write cursor of sub-bucket j in a register, positions come from
  // ballots -- no shared memory, no barriers, no atomics, and the eight warps of a CTA keep eight buckets'
  // loads (local HBM or NVLink) in flight.
  constexpr int U = 4;                 // elements per lane and step
  const int d2 = ga.d2, digit_pos = ga.digit_pos;
  const uint32_t n_src = ga.n_src, nb = ga.nb, lo = ga.lo, hi = ga.hi;
  const uint32_t nbins = 1u << d2, mask = nbins - 1u;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * NT + threadIdx.x) >> 5, nwarps = (gridDim.x * NT) >> 5;
  Elem* __restrict__ out = ga.out;
  for (uint32_t b = lo + warp; b < hi; b += nwarps) {
    // ---- sub-bucket sizes
    uint32_t mine = 0;                 // lane j: size of sub-bucket j
    if (d2 == 0) {
      for (uint32_t s = 0; s < n_src; s++) mine += ga.sizes_all[(size_t)s * nb + b];  // only lane 0's copy is used
    } else if (ga.sub_ptrs) {
      if (lane < nbins)
        for (uint32_t s = 0; s < n_src; s++) mine += ga.sub_ptrs[s][((size_t)b << d2) + lane];
    } else if (ga.sub_sizes) {
      const size_t row = (size_t)(hi - lo) << d2;
      if (lane < nbins)
        for (uint32_t s = 0; s < n_src; s++) mine += ga.sub_sizes[(size_t)s * row + (((size_t)(b - lo)) << d2) + lane];
    } else {
      for (uint32_t s = 0; s < n_src; s++) {
        const uint32_t n = ga.sizes_all[(size_t)s * nb + b];
        const Elem* src = ga.src_base[s] + (ga.seg_off ? ga.seg_off[s] : 0ull) + ga.piece_off[(size_t)s * (nb + 1) + b];
        for (uint32_t i0 = 0; i0 < n; i0 += 32 * U) {
          uint32_t d[U];
#pragma unroll
          for (int u = 0; u < U; u++) {
            const uint32_t i = i0 + u * 32 + lane;
            d[u] = i < n ? split_digit(src[i], digit_pos, mask) : 0xFFFFFFFFu;
          }
          for (uint32_t j = 0; j < nbins; j++) {
            uint32_t cnt = 0;
#pragma unroll
            for (int u = 0; u < U; u++) cnt += __popc(__ballot_sync(0xffffffffu, d[u] == j));
            if (lane == j) mine += cnt;
          }
        }
      }
    }
    if (lane >= nbins) mine = 0;
    // exclusive scan over the lanes -> start of every sub-bucket, relative to the bucket
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if ((int)lane >= o) incl += v;
    }
    uint32_t cur = incl - mine;        // lane j: next free slot of sub-bucket j
    const unsigned long long base_b = ga.bofs_coarse[b] - ga.coarse_base;
    if (lane < nbins) {
      const size_t f = ((size_t)b << d2) | lane;
      ga.bsize_fine[f] = mine;
      ga.bofs_fine[f] = base_b + cur;
    }
    // ---- place.  32-bit elements are fetched 16 bytes per lane (512 bytes per warp instruction: NVLink
    // and HBM both like long requests); a scalar step first brings the piece to 16-byte alignment.
    for (uint32_t s = 0; s < n_src; s++) {
      const uint32_t n = ga.sizes_all[(size_t)s * nb + b];
      const Elem* src = ga.src_base[s] + (ga.seg_off ? ga.seg_off[s] : 0ull) + ga.piece_off[(size_t)s * (nb + 1) + b];
      uint32_t head = 0;
      if constexpr (sizeof(Elem) == 4) {
        head = (uint32_t)((16u - ((uint32_t)(uintptr_t)src & 15u)) & 15u) >> 2;
        if (head > n) head = n;
      }
      for (uint32_t i0 = 0; i0 < n; i0 += (i0 < head ? head : 32 * U)) {
        Elem e[U];
        uint32_t d[U], pos[U];
#pragma unroll
        for (int u = 0; u < U; u++) { d[u] = 0xFFFFFFFFu; pos[u] = 0; e[u] = Elem{}; }
        if (sizeof(Elem) == 4 && i0 < head) {            // alignment step: lanes 0 .. head-1, one element each
          if (lane < head) { e[0] = src[lane]; d[0] = split_digit(e[0], digit_pos, mask); }
        } else if constexpr (sizeof(Elem) == 4) {        // lane takes elements i0 + 4*lane .. +3
          const uint32_t i = i0 + 4 * lane;
          if (i + 3 < n) {
            const uint4 v = *reinterpret_cast<const uint4*>(src + i);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int u = 0; u < U; u++) { memcpy(&e[u], &w[u], 4); d[u] = split_digit(e[u], digit_pos, mask); }
          } else {
#pragma unroll
            for (int u = 0; u < U; u++)
              if (i + u < n) { e[u] = src[i + u]; d[u] = split_digit(e[u], digit_pos, mask); }
          }
        } else {
#pragma unroll
          for (int u = 0; u < U; u++) {
            const uint32_t i = i0 + u * 32 + lane;
            if (i < n) { e[u] = src[i]; d[u] = split_digit(e[u], digit_pos, mask); }
          }
        }
        for (uint32_t j = 0; j < nbins; j++) {
          uint32_t base = __shfl_sync(0xffffffffu, cur, j), tot = 0;
#pragma unroll
          for (int u = 0; u < U; u++) {
            const uint32_t m = __ballot_sync(0xffffffffu, d[u] == j);
            if (d[u] == j) pos[u] = base + tot + __popc(m & ((1u << lane) - 1u));
            tot += __popc(m);
          }
          if (lane == j) cur += tot;
        }
#pragma unroll
        for (int u = 0; u < U; u++)
          if (d[u] != 0xFFFFFFFFu) out[base_b + pos[u]] = split_strip(e[u], digit_pos);
      }
    }
  }
}

// ---------------------------------------------------------------- the gather, pipelined through shared memory
// Same contract as k_gather_split (sub-bucket sizes known: d2 == 0, ga.sub_ptrs or ga.sub_sizes), but the pieces
// reach the warp through cp.async (LDGSTS): every warp owns two stages of GS_CHUNK elements in shared memory and
// always has the NEXT chunk of its bucket's piece stream -- piece after piece, source after source -- in flight
// while it splits the current one.  In the round-1 kernel a lane had ONE 16-byte load outstanding and sat through
// an NVLink round trip (2-3 us) per 512 bytes per warp: 0.46-0.55 of the link at 8 GPUs.  Here a warp keeps
// 1-6 KB in flight without holding it in registers, the copies need no alignment (element-sized cp.async), and
// loading overlaps the ballots and the stores.
template <typename Elem> struct GsChunk { static constexpr int N = sizeof(Elem) == 4 ? 512 : 256; };   // elements per stage (2 KB+)
__device__ __forceinline__ void cp_async_elem(uint32_t smem_dst, const uint32_t* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(src) : "memory");
}
template <int W>
__device__ __forceinline__ void cp_async_elem(uint32_t smem_dst, const Key<W>* src) {
#pragma unroll
  for (int i = 0; i < W; i++)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst + 8 * i), "l"(&src->w[i]) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <typename Elem, int NT>
__global__ void __launch_bounds__(NT) k_gather_split2(const GatherArgs<Elem> ga) {
  extern __shared__ __align__(16) unsigned char gs_raw[];
  constexpr int U = 4;                 // elements per lane and ballot round
  constexpr int GS_CHUNK = GsChunk<Elem>::N;
  const int d2 = ga.d2, digit_pos = ga.digit_pos;
  const uint32_t n_src = ga.n_src, nb = ga.nb, lo = ga.lo, hi = ga.hi;
  const uint32_t nbins = 1u << d2, mask = nbins - 1u;
  const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t warp = (blockIdx.x * NT + threadIdx.x) >> 5, nwarps = (gridDim.x * NT) >> 5;
  Elem* stage = reinterpret_cast<Elem*>(gs_raw) + (size_t)wib * 2 * GS_CHUNK;   // this warp's two stages
  const uint32_t stage_a = smem_u32(stage);
  Elem* __restrict__ out = ga.out;
  for (uint32_t b = lo + warp; b < hi; b += nwarps) {
    // ---- sub-bucket sizes -> write cursors (lane j: sub-bucket j)
    uint32_t mine = 0;
    if (d2 == 0) {
      for (uint32_t s = 0; s < n_src; s++) mine += ga.sizes_all[(size_t)s * nb + b];
    } else if (ga.sub_ptrs) {
      if (lane < nbins)
        for (uint32_t s = 0; s < n_src; s++) mine += ga.sub_ptrs[s][((size_t)b << d2) + lane];
    } else {
      const size_t row = (size_t)(hi - lo) << d2;
      if (lane < nbins)
        for (uint32_t s = 0; s < n_src; s++) mine += ga.sub_sizes[(size_t)s * row + (((size_t)(b - lo)) << d2) + lane];
    }
    if (lane >= nbins) mine = 0;
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if ((int)lane >= o) incl += v;
    }
    uint32_t cur = incl - mine;
    const unsigned long long base_b = ga.bofs_coarse[b] - ga.coarse_base;
    if (lane < nbins) {
      const size_t f = ((size_t)b << d2) | lane;
      ga.bsize_fine[f] = mine;
      ga.bofs_fine[f] = base_b + cur;
    }
    // ---- the bucket's piece stream: a load cursor one chunk ahead of the split
    uint32_t ls = 0, loff = 0, ln = 0;
    const Elem* lsrc = nullptr;
    auto next_piece = [&]() {   // first non-empty piece from source ls on (warp-uniform)
      while (ls < n_src) {
        ln = ga.sizes_all[(size_t)ls * nb + b];
        if (ln) { lsrc = ga.src_base[ls] + (ga.seg_off ? ga.seg_off[ls] : 0ull) + ga.piece_off[(size_t)ls * (nb + 1) + b]; return; }
        ls++;
      }
    };
    auto issue = [&](uint32_t st) -> uint32_t {   // start the copy of the next chunk into stage st; -> its length (0: stream over)
      if (ls >= n_src) return 0u;
      const uint32_t cnt = ln - loff < (uint32_t)GS_CHUNK ? ln - loff : (uint32_t)GS_CHUNK;
      const Elem* src = lsrc + loff;
      const uint32_t dst = stage_a + st * (uint32_t)(GS_CHUNK * sizeof(Elem));
#pragma unroll
      for (int u = 0; u < GS_CHUNK / 32; u++) {
        const uint32_t i = u * 32 + lane;
        if (i < cnt) cp_async_elem(dst + i * (uint32_t)sizeof(Elem), src + i);
      }
      cp_async_commit();
      loff += cnt;
      if (loff == ln) { ls++; loff = 0; next_piece(); }
      return cnt;
    };
    next_piece();
    uint32_t st = 0;
    uint32_t cnt_cur = issue(0);
    while (cnt_cur) {
      const uint32_t cnt_next = issue(st ^ 1u);
      if (cnt_next) cp_async_wait<1>(); else cp_async_wait<0>();
      __syncwarp();
      const Elem* sm = stage + (size_t)st * GS_CHUNK;
      for (uint32_t i0 = 0; i0 < cnt_cur; i0 += 32 * U) {
        Elem e[U];
        uint32_t d[U], pos[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const uint32_t i = i0 + u * 32 + lane;
          d[u] = 0xFFFFFFFFu; pos[u] = 0;
          if (i < cnt_cur) { e[u] = sm[i]; d[u] = split_digit(e[u], digit_pos, mask); } else e[u] = Elem{};
        }
        for (uint32_t j = 0; j < nbins; j++) {
          uint32_t base = __shfl_sync(0xffffffffu, cur, j), tot = 0;
#pragma unroll
          for (int u = 0; u < U; u++) {
            const uint32_t m = __ballot_sync(0xffffffffu, d[u] == j);
            if (d[u] == j) pos[u] = base + tot + __popc(m & ((1u << lane) - 1u));
            tot += __popc(m);
          }
          if (lane == j) cur += tot;
        }
#pragma unroll
        for (int u = 0; u < U; u++)
          if (d[u] != 0xFFFFFFFFu) out[base_b + pos[u]] = split_strip(e[u], digit_pos);
      }
      __syncwarp();   // every lane is done with stage st before a later copy lands in it
      st ^= 1u;
      cnt_cur = cnt_next;
    }
  }
}

// ---------------------------------------------------------------- sharded counting: the plan of an exchange, on the device
// u64 bucket sizes of this rank's partition -> u32 (what travels in the all-gather); flag |= 1 if one does not fit
__global__ void k_sizes32(const unsigned long long* __restrict__ in, uint32_t nb, uint32_t* __restrict__ out,
                          unsigned long long* __restrict__ flag) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  const unsigned long long v = in[b];
  if (v >= (1ull << 31)) { atomicOr(flag, 1ull); out[b] = 0; }
  else out[b] = (uint32_t)v;
}
// merged size of every bucket over the sources; flag |= 2 if one reaches 2^32.  cost32 (may be null): what
// counting the bucket costs, in key units -- its keys plus `bucket_cost` for being a bucket at all.
__global__ void k_total_sizes(const uint32_t* __restrict__ sizes_all, uint32_t n_src, uint32_t nb, uint32_t* __restrict__ tot32,
                              unsigned long long* __restrict__ flag, uint32_t* __restrict__ cost32, uint32_t bucket_cost) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  unsigned long long t = 0;
  for (uint32_t s = 0; s < n_src; s++) t += sizes_all[(size_t)s * nb + b];
  if (t >= (1ull << 32)) { atomicOr(flag, 2ull); t = 0; }
  tot32[b] = (uint32_t)t;
  if (cost32) {
    const unsigned long long c = t ? t + bucket_cost : 0ull;
    cost32[b] = c >= (1ull << 32) ? 0xFFFFFFFFu : (uint32_t)c;
  }
}
// Balanced contiguous bucket ranges from the exclusive prefix S[nb + 1] of the buckets' weights (their merged sizes,
// or their costs): range r ends after the first bucket whose cumulative weight exceeds total * (r + 1) / world (the
// rule of dist.balanced_splitters).  plan[0 .. world] = bounds, plan[world + 1 .. 2 world + 1] = E (the prefix of the
// merged SIZES) at the bounds, plan[2 world + 2 ..] = own[] at the bounds (the calling rank's own prefix: how much of
// each range it holds itself).  One thread per bound.
// bound r of `world` ranges over nb buckets with weight prefix S[nb + 1]  (host-callable: the CPU suite checks the rule)
APGK_HD uint32_t splitter_bound(const unsigned long long* S, uint32_t nb, uint32_t world, uint32_t r) {
  if (r == 0) return 0;
  if (r >= world) return nb;
  const unsigned long long total = S[nb];
  const unsigned long long target = (unsigned long long)(((unsigned __int128)total * r) / world);
  // smallest b in [0, nb] with S[b + 1] > target  (S[nb + 1] := infinity)
  uint32_t lo = 0, hi = nb;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (S[mid + 1] > target) hi = mid; else lo = mid + 1;
  }
  return lo;
}
__global__ void k_splitters(const unsigned long long* __restrict__ S, const unsigned long long* __restrict__ E, uint32_t nb, uint32_t world,
                            const unsigned long long* __restrict__ own, unsigned long long* __restrict__ plan) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > world) return;
  const uint32_t bound = splitter_bound(S, nb, world, r);
  plan[r] = bound;
  plan[world + 1 + r] = E[bound];
  plan[2 * (world + 1) + r] = own[bound];
}
// out[i] = sum over ranks of in[r][i]  (in-process form of the spectrum all-reduce)
__global__ void k_sum_ranks(const unsigned long long* const* __restrict__ in, uint32_t n_ranks, uint64_t n, unsigned long long* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long t = 0;
  for (uint32_t r = 0; r < n_ranks; r++) t += in[r][i];
  out[i] = t;
}
__global__ void k_max_ranks(const unsigned long long* const* __restrict__ in, uint32_t n_ranks, uint64_t n, unsigned long long* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long t = 0;
  for (uint32_t r = 0; r < n_ranks; r++) t = in[r][i] > t ? in[r][i] : t;
  out[i] = t;
}

// ---------------------------------------------------------------- compaction: temp records -> final table
// One warp per bucket.  Temp keys / counts live at element offset bofs[b] of the temp buffers.
// Guarded form (total != null): the host launched this without knowing the record count; when *total exceeds
// the buffers' capacity nothing is written and *overflow is raised (the host grows the buffers and runs it again).
template <int W>
__global__ void k_compact(const Key<W>* __restrict__ tmp_keys, const uint32_t* __restrict__ tmp_cnt,
                          const unsigned long long* __restrict__ bofs,
                          const unsigned long long* __restrict__ out_off, uint32_t nb, Key<W>* __restrict__ out_keys,
                          uint32_t* __restrict__ out_cnt, const unsigned long long* __restrict__ total,
                          unsigned long long capacity, unsigned long long* __restrict__ overflow) {
  if (total && *total > capacity) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 1ull;
    return;
  }
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t b = warp; b < nb; b += nwarps) {
    const unsigned long long o0 = out_off[b], nd = out_off[b + 1] - o0;
    if (!nd) continue;
    const unsigned long long src = bofs[b];
    for (unsigned long long j = lane; j < nd; j += 32) {
      out_keys[o0 + j] = tmp_keys[src + j];
      out_cnt[o0 + j] = tmp_cnt[src + j];
    }
  }
}

// ---------------------------------------------------------------- lookups
template <int W>
APGK_HD Key<W> key_revcomp(const Key<W>& x, int K) {
  const int topbits = 2 * K - 64 * (W - 1);
  Key<W> y;
#pragma unroll
  for (int i = 0; i < W; i++) y.w[i] = ~x.w[i];
  y.w[0] &= lowmask64(topbits);
  // reverse the 2-bit groups of the 64W-bit value, then shift right by 64W - 2K
  uint64_t rm[W];
#pragma unroll
  for (int i = 0; i < W; i++) rm[i] = swap_pairs(brev64(y.w[W - 1 - i]));
  const int s = 64 * W - 2 * K;
  Key<W> r;
#pragma unroll
  for (int i = 0; i < W; i++) {
    uint64_t v = rm[i] >> s;
    if (i > 0 && s > 0) v |= rm[i - 1] << (64 - s);
    r.w[i] = v;
  }
  return r;
}
template <int W>
APGK_HD Key<W> key_canonical(const Key<W>& x, int K) {
  Key<W> rc = key_revcomp(x, K);
  return key_less(rc, x) ? rc : x;
}

template <int W>
struct FreqTable {
  const Key<W>* keys;               // n_distinct, ascending
  const uint32_t* counts;           // n_distinct
  const unsigned long long* index;  // [nb+1] first record of each prefix bucket
  uint32_t nb;
  int prefix_pos, prefix_len, pad;  // bucket = digits of the key's leading P bits
  int D1;
};

// Index of canonical k-mer c in the table, ~0 if absent.  The prefix index narrows the search to one
// level-1 bucket; inside it the keys are close to uniformly spread over the remainder space, so the
// search starts at the interpolated slot (next 16 key bits), brackets the answer by galloping (8, 16,
// 32 ... slots) and finishes with a binary search inside the bracket: ~3 dependent DRAM sectors per
// query instead of ~10 for a plain binary search over a ~600-key bucket.  Correct for any key
// distribution (a skewed bucket only gallops further).  Host-callable for the CPU test of the search.
template <int W>
APGK_HD unsigned long long table_find_index(const FreqTable<W>& t, const Key<W>& c) {
  // prefix bucket = (digit0 << D1) | digit1 = bits [prefix_pos, prefix_pos + prefix_len) of the virtual key
  const uint32_t b = digit_of(c, t.prefix_pos, t.prefix_len, t.pad);
  const unsigned long long lo0 = t.index[b], hi0 = t.index[b + 1];
  unsigned long long lo = lo0, hi = hi0;  // invariant: keys below lo are < c, keys from hi on are >= c
  if (hi - lo > 16) {
    const int fb = t.prefix_pos < 16 ? t.prefix_pos : 16;
    const unsigned long long frac = digit_of(c, t.prefix_pos - fb, fb, t.pad);
    const unsigned long long g = lo + (((hi - lo) * frac) >> fb);  // lo0 <= g < hi0
    unsigned long long step = 8;
    if (key_less(t.keys[g], c)) {
      lo = g + 1;
      for (;;) {
        const unsigned long long h = hi0 - lo > step ? lo + step : hi0;
        if (h == lo) { hi = lo; break; }
        if (key_less(t.keys[h - 1], c)) {
          lo = h;
          if (h == hi0) { hi = h; break; }
          step <<= 1;
        } else { hi = h - 1; break; }
      }
    } else {
      hi = g;
      for (;;) {
        if (hi == lo0) { lo = lo0; break; }
        const unsigned long long l = hi - lo0 > step ? hi - step : lo0;
        if (key_less(t.keys[l], c)) { lo = l + 1; break; }
        hi = l;
        step <<= 1;
      }
    }
  }
  while (lo < hi) {
    const unsigned long long mid = (lo + hi) >> 1;
    if (key_less(t.keys[mid], c)) lo = mid + 1; else hi = mid;
  }
  if (lo < hi0 && key_eq(t.keys[lo], c)) return lo;
  return ~0ull;
}
template <int W>
APGK_HD uint32_t table_find(const FreqTable<W>& t, const Key<W>& c) {
  const unsigned long long i = table_find_index(t, c);
  return i == ~0ull ? 0u : t.counts[i];
}

template <int W>
__global__ void k_lookup(FreqTable<W> t, const Key<W>* __restrict__ q, uint64_t nq, int K, int canonicalise,
                         uint32_t* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  Key<W> c = q[i];
  if (canonicalise) c = key_canonical(c, K);
  out[i] = table_find(t, c);
}

// count of the canonical k-mer starting at every base of the read store
// (0xFFFFFFFF where the window leaves its read).
template <int W, int NT>
__global__ void __launch_bounds__(NT) k_read_freqs(ReadStore rs, FreqTable<W> t, uint64_t first_base, uint64_t n_bases,
                                                   uint32_t* __restrict__ out) {
  const uint64_t p = (first_base & ~15ull) + ((uint64_t)blockIdx.x * NT + threadIdx.x) * POS_PER_THREAD;
  if (p >= first_base + n_bases) return;
  const uint32_t valid = window_valid_mask16(rs.starts32, p, rs.K, rs.total_bases);
  uint32_t res[POS_PER_THREAD];
#pragma unroll
  for (int j = 0; j < POS_PER_THREAD; j++) res[j] = 0xFFFFFFFFu;
  if (valid) {
    Window16<W> win;
    load_window16<W>(rs.bases32, p, rs.K, win);
    extract16<W>(win, rs.K, [&](int j, const Key<W>& c, bool) {
      if ((valid >> j) & 1u) res[j] = table_find(t, c);
    });
  }
#pragma unroll
  for (int j = 0; j < POS_PER_THREAD; j++) {
    const uint64_t q = p + j;
    if (q >= first_base && q < first_base + n_bases) out[q - first_base] = res[j];
  }
}

// ---------------------------------------------------------------- read store maintenance
// Append nbits of a bit stream (src, starting at bit src_bit0) to dst at bit dst_bit0.
// One thread per destination 64-bit word; partial first/last words are OR-ed in
// (destination beyond the current end must be zero).
__global__ void k_append_bits(const uint64_t* __restrict__ src, uint64_t src_bit0, uint64_t* __restrict__ dst,
                              uint64_t dst_bit0, uint64_t nbits) {
  const uint64_t w0 = dst_bit0 >> 6, w1 = (dst_bit0 + nbits + 63) >> 6;
  const uint64_t w = w0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= w1) return;
  // destination bits [lo, hi) of this word, absolute
  uint64_t lo = w << 6, hi = lo + 64;
  if (lo < dst_bit0) lo = dst_bit0;
  if (hi > dst_bit0 + nbits) hi = dst_bit0 + nbits;
  const uint64_t sb = src_bit0 + (lo - dst_bit0);  // source bit matching destination bit lo
  const uint64_t si = sb >> 6;
  const uint32_t ss = (uint32_t)(sb & 63);
  uint64_t v = src[si] >> ss;
  if (ss) v |= src[si + 1] << (64 - ss);  // src is padded by one word
  const uint32_t len = (uint32_t)(hi - lo);
  v &= lowmask64((int)len);
  v <<= (lo & 63);
  if (len == 64) dst[w] = v; else atomicOr((unsigned long long*)&dst[w], (unsigned long long)v);
}

// starts bitmap from read offsets: bit (dst_base0 + off[r] - off0) for every read r
__global__ void k_mark_starts(const uint64_t* __restrict__ off, uint64_t n_reads, uint64_t off0, uint64_t dst_base0,
                              uint32_t* __restrict__ starts32) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  const uint64_t q = dst_base0 + (off[r] - off0);
  atomicOr(&starts32[q >> 5], 1u << (q & 31));
}
__global__ void k_mark_starts_uniform(uint64_t n_reads, uint32_t read_len, uint64_t dst_base0,
                                      uint32_t* __restrict__ starts32) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  const uint64_t q = dst_base0 + r * read_len;
  atomicOr(&starts32[q >> 5], 1u << (q & 31));
}

// ---------------------------------------------------------------- synthetic reads (SURVEY.md section 8d generator)
struct SynthParams {
  uint64_t genome_len;
  uint64_t seed_g, seed_p, seed_q, seed_r, seed_e;
  uint32_t read_len;
  uint32_t err_per_200;
};
APGK_HD uint32_t synth_genome_base(const SynthParams& p, uint64_t i) {
  const uint64_t b = i / 5000u;
  if (b > 0 && sm64(p.seed_p ^ b) % 50u == 0) {
    const uint64_t src = sm64(p.seed_q ^ b) % b;
    i = src * 5000u + i % 5000u;
  }
  return (uint32_t)(sm64(p.seed_g ^ i) & 3u);
}
struct SynthRead {
  uint64_t start;
  bool rev;
};
APGK_HD SynthRead synth_read_info(const SynthParams& p, uint64_t r) {
  SynthRead sr;
  sr.start = sm64(p.seed_r ^ (2 * r)) % (p.genome_len - p.read_len + 1);
  sr.rev = (sm64(p.seed_r ^ (2 * r + 1)) >> 63) != 0;
  return sr;
}
APGK_HD uint32_t synth_read_base(const SynthParams& p, const SynthRead& sr, uint64_t r, uint32_t j) {
  const uint32_t L = p.read_len;
  uint32_t b = sr.rev ? 3u - synth_genome_base(p, sr.start + (L - 1 - j)) : synth_genome_base(p, sr.start + j);
  if (p.err_per_200) {
    const uint64_t e = sm64(p.seed_e ^ (r * (uint64_t)L + j));
    if ((e >> 32) % 200u < p.err_per_200) b = (b + 1u + (uint32_t)((e >> 8) % 3u)) & 3u;
  }
  return b;
}
// 16 bases (one store word) starting at base q of the concatenated reads r0, r0+1, ...
APGK_HD uint32_t synth_word(const SynthParams& sp, uint64_t r0, uint64_t q, uint64_t nb) {
  uint32_t v = 0;
  uint64_t r = q / sp.read_len;
  uint32_t j = (uint32_t)(q % sp.read_len);
  SynthRead sr = synth_read_info(sp, r0 + r);
  for (int t = 0; t < 16 && q < nb; t++, q++) {
    v |= synth_read_base(sp, sr, r0 + r, j) << (2 * t);
    if (++j == sp.read_len) {
      j = 0;
      r++;
      sr = synth_read_info(sp, r0 + r);
    }
  }
  return v;
}
// one thread per 32-bit word (16 bases) of the store, starting at base dst_base0 (multiple of 16)
__global__ void k_synth(SynthParams sp, uint64_t r0, uint64_t n_reads, uint64_t dst_base0, uint32_t* __restrict__ bases32) {
  const uint64_t nb = n_reads * sp.read_len;
  const uint64_t wi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (wi * 16 >= nb) return;
  bases32[(dst_base0 >> 4) + wi] = synth_word(sp, r0, wi * 16, nb);
}

}  // namespace apgk
