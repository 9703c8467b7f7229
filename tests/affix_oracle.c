/*
 * tests/affix_oracle.c -- CPU oracle "A" for the k-mer AFFIXES (apgk_build_affixes).  TEST INFRASTRUCTURE.
 *
 * Restates the definition in include/apgk.h on the same roll + binary search shape as oracle/kmer_oracle.c's
 * oracle_read_freqs / oracle_occurrences (bases A=0 C=1 G=2 T=3, 2-bit packed little-endian, a k-mer = the 2K-bit
 * integer with its first base most significant in W = ceil(2K/64) words, most significant word first):
 *   window x at base p of a read, L = base p-1 (none at the read's first base), R = base p+K (none past its end);
 *   x < rc(x): pre(x) |= L, suf(x) |= R;  x > rc(x): pre(rc(x)) |= comp(R), suf(rc(x)) |= comp(L);  x == rc(x): both.
 * Byte of a k-mer: bit b = base b precedes, bit 4+b = base b follows.
 * Every OpenMP thread ORs into a private byte array; the arrays are OR-reduced at the end.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define MAXW 3

static inline uint32_t base_at(const uint8_t* packed, uint64_t q) { return (packed[q >> 2] >> ((q & 3) * 2)) & 3u; }

static inline int cmp_words(const uint64_t* a, const uint64_t* b, int W) {
  for (int i = 0; i < W; i++) {
    if (a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
  }
  return 0;
}

/* out[i] = affix byte of kmers[i] (sorted, distinct, canonical).  0 on success, -3 when a window's canonical k-mer is
 * missing from `kmers`, -2 when memory runs out. */
int oracle_affixes(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, const uint64_t* kmers,
                   uint64_t n_distinct, uint8_t* out) {
  if (K < 1 || K > 32 * MAXW) return -1;
  const int W = (2 * K + 63) / 64;
  const int topbits = 2 * K - 64 * (W - 1);
  const uint64_t topmask = topbits == 64 ? ~0ull : ((1ull << topbits) - 1);
  int status = 0;
  memset(out, 0, n_distinct);
#pragma omp parallel
  {
    uint8_t* mine = (uint8_t*)calloc(n_distinct + 1, 1);
    int err = mine ? 0 : -2;
#pragma omp for schedule(dynamic, 64)
    for (int64_t r = 0; r < (int64_t)n_reads; r++) {
      const uint64_t b0 = off[r], b1 = off[r + 1];
      if (err || b1 - b0 < (uint64_t)K) continue;
      uint64_t fw[MAXW] = {0, 0, 0}, rc[MAXW] = {0, 0, 0};
      for (uint64_t q = b0; q < b1 && !err; q++) {
        const uint32_t b = base_at(packed, q);
        for (int i = 0; i < W - 1; i++) fw[i] = (fw[i] << 2) | (fw[i + 1] >> 62);   /* forward roll */
        fw[W - 1] = (fw[W - 1] << 2) | b;
        fw[0] &= topmask;
        for (int i = W - 1; i > 0; i--) rc[i] = (rc[i] >> 2) | (rc[i - 1] << 62);   /* reverse-complement roll */
        rc[0] = (rc[0] >> 2) | ((uint64_t)(3u - b) << (topbits - 2));
        if (q + 1 - b0 < (uint64_t)K) continue;
        const uint64_t p = q + 1 - (uint64_t)K;
        const int has_l = p > b0, has_r = q + 1 < b1;
        const uint32_t L = has_l ? base_at(packed, p - 1) : 0, R = has_r ? base_at(packed, q + 1) : 0;
        const int cmp = cmp_words(fw, rc, W);
        uint32_t pre = 0, suf = 0;
        if (cmp <= 0) {   /* read forward (a palindrome both ways) */
          if (has_l) pre |= 1u << L;
          if (has_r) suf |= 1u << R;
        }
        if (cmp >= 0) {   /* read as its reverse complement */
          if (has_r) pre |= 1u << (3u - R);
          if (has_l) suf |= 1u << (3u - L);
        }
        const uint64_t* c = cmp <= 0 ? fw : rc;
        uint64_t lo = 0, hi = n_distinct;
        while (lo < hi) {
          const uint64_t mid = (lo + hi) / 2;
          if (cmp_words(kmers + mid * W, c, W) < 0) lo = mid + 1; else hi = mid;
        }
        if (lo >= n_distinct || cmp_words(kmers + lo * W, c, W) != 0) { err = -3; break; }
        mine[lo] |= (uint8_t)(pre | (suf << 4));
      }
    }
#pragma omp critical
    {
      if (err) status = err;
      else for (uint64_t i = 0; i < n_distinct; i++) out[i] |= mine[i];
    }
    free(mine);
  }
  return status;
}
