/*
 * oracle/kmer_oracle.c -- CPU oracle "A" for the k-mer spectrum hot path.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this file's
 * library.  Nothing under allpathslg_b200/ may call it.
 *
 * PARITY UNPINNED.  /root/reference was empty when this was written
 * (SURVEY.md section 0), so no reference file:line can be cited and no
 * reference golden vector exists.  This file restates the DEFINITION in
 * SURVEY.md section 8 ("Definition the whole table rests on"), which is the
 * survey's recollection of what ALLPATHS-LG's k-mer layer computes
 * (kmers/SortKmers, kmers/KmerParcels, kmers/KmerSpectra, kmers/naif_kmer --
 * names from BASELINE.json / recollection, unverified):
 *
 *   - bases A=0 C=1 G=2 T=3, complement(b) = 3-b;
 *   - reads are 2-bit packed, base i of the stream at bits [2i, 2i+2) of the
 *     byte stream (little-endian within a byte: base 0 in bits 0..1);
 *   - read r covers bases off[r] .. off[r+1]-1 and yields max(0, L-K+1) k-mers;
 *   - a k-mer is the 2K-bit integer with its FIRST base most significant;
 *     canonical(x) = min(x, revcomp(x)) as unsigned integers; a palindrome
 *     counts once per instance;
 *   - count[c] = number of instances with canonical form c (uint64, uncapped);
 *   - spectrum[f] = number of distinct c with count[c] == f, f >= 1.
 *
 * It is cross-checked against an independently written oracle "B"
 * (oracle/oracle_b.py, string/dict based) and against hand-computed
 * known-answer vectors in tests/golden/.
 *
 * Algorithm (deliberately different from the GPU pipeline's smem radix sort,
 * but the same shape as the reference's "passes over k-mer space" idea):
 *   1. each thread rolls fw / rc over its reads, 2 bits per base, and counts
 *      canonical k-mers per bucket (top bits of the k-mer);
 *   2. prefix sums give every (thread, bucket) a private output range;
 *   3. second roll scatters the k-mers;
 *   4. buckets are sorted independently (LSD byte radix for 1-word k-mers,
 *      qsort for multi-word) and run-length counted.
 *
 * K-mers are stored as W = ceil(2K/64) uint64 words, MOST significant word
 * first, value right-aligned (top word holds the 2K - 64(W-1) high bits).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define MAXW 4

/* ------------------------------------------------------------------ hashing
 * splitmix64 finaliser used by the synthetic read generator (SURVEY 8d). */
static inline uint64_t sm64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

/* ------------------------------------------------------------------ generator
 * Synthetic reads, pure function of (seeds, read index, base index):
 *   genome base i : block b = i / 5000; if b > 0 and sm64(seed_p ^ b) % 50 == 0
 *                   the block is a planted repeat of block src = sm64(seed_q ^ b) % b
 *                   (raw bases of the source block); base = sm64(seed_g ^ i') & 3.
 *   read r        : start = sm64(seed_r ^ 2r) % (G - L + 1);
 *                   reverse strand iff bit 63 of sm64(seed_r ^ (2r+1));
 *                   base j = genome(start + j) or 3 - genome(start + L-1-j);
 *                   e = sm64(seed_e ^ (r*L + j)); if (e >> 32) % 200 == 0 the base
 *                   becomes (base + 1 + (e >> 8) % 3) & 3   (0.5 % substitutions).
 */
typedef struct {
  uint64_t genome_len;
  uint64_t seed_g, seed_p, seed_q, seed_r, seed_e;
  uint32_t read_len;
  uint32_t err_per_200; /* 1 -> 0.5 %; 0 -> no errors */
} synth_params;

static inline uint32_t genome_base(const synth_params* p, uint64_t i) {
  uint64_t b = i / 5000u;
  if (b > 0 && sm64(p->seed_p ^ b) % 50u == 0) {
    uint64_t src = sm64(p->seed_q ^ b) % b;
    i = src * 5000u + i % 5000u;
  }
  return (uint32_t)(sm64(p->seed_g ^ i) & 3u);
}

static inline uint32_t read_base(const synth_params* p, uint64_t r, uint32_t j) {
  uint32_t L = p->read_len;
  uint64_t start = sm64(p->seed_r ^ (2 * r)) % (p->genome_len - L + 1);
  int rev = (int)(sm64(p->seed_r ^ (2 * r + 1)) >> 63);
  uint32_t b = rev ? 3u - genome_base(p, start + (L - 1 - j)) : genome_base(p, start + j);
  if (p->err_per_200) {
    uint64_t e = sm64(p->seed_e ^ (r * (uint64_t)L + j));
    if ((e >> 32) % 200u < p->err_per_200) b = (b + 1u + (uint32_t)((e >> 8) % 3u)) & 3u;
  }
  return b;
}

/* Fill packed[] (caller-zeroed or not; fully overwritten, size ceil(n*L/4)
 * rounded up to 8 bytes) with reads [r0, r0+n) back to back. */
void oracle_synth_reads(const synth_params* p, uint64_t r0, uint64_t n, uint8_t* packed) {
  uint64_t nb = n * (uint64_t)p->read_len;
  uint64_t nwords = (nb + 31) / 32;
  uint64_t* w = (uint64_t*)packed;
#pragma omp parallel for schedule(static)
  for (int64_t wi = 0; wi < (int64_t)nwords; wi++) {
    uint64_t v = 0;
    for (int t = 0; t < 32; t++) {
      uint64_t q = (uint64_t)wi * 32 + t;
      if (q >= nb) break;
      uint64_t r = r0 + q / p->read_len;
      uint32_t j = (uint32_t)(q % p->read_len);
      v |= (uint64_t)read_base(p, r, j) << (2 * t);
    }
    w[wi] = v;
  }
}

/* ------------------------------------------------------------------ k-mer roll */
typedef struct { uint64_t w[MAXW]; } kw_t;

static inline uint32_t get_base(const uint8_t* packed, uint64_t q) {
  return (packed[q >> 2] >> ((q & 3) * 2)) & 3u;
}

/* fw = (fw << 2 | b) & mask  over W words (w[0] most significant) */
static inline void roll_fw(uint64_t* fw, int W, uint64_t topmask, uint32_t b) {
  for (int i = 0; i < W - 1; i++) fw[i] = (fw[i] << 2) | (fw[i + 1] >> 62);
  fw[W - 1] = (fw[W - 1] << 2) | b;
  fw[0] &= topmask;
}
/* rc = (rc >> 2) | (3-b) << 2(K-1) */
static inline void roll_rc(uint64_t* rc, int W, int topshift, uint32_t b) {
  for (int i = W - 1; i > 0; i--) rc[i] = (rc[i] >> 2) | (rc[i - 1] << 62);
  rc[0] = (rc[0] >> 2) | ((uint64_t)(3u - b) << topshift);
}
static inline int cmp_w(const uint64_t* a, const uint64_t* b, int W) {
  for (int i = 0; i < W; i++) {
    if (a[i] < b[i]) return -1;
    if (a[i] > b[i]) return 1;
  }
  return 0;
}

typedef void (*emit_fn)(void* ctx, const uint64_t* canon);

/* Roll over reads [r_lo, r_hi) and emit every canonical k-mer. */
static void roll_reads(const uint8_t* packed, const uint64_t* off, uint64_t r_lo, uint64_t r_hi, int K, int W,
                       emit_fn emit, void* ctx) {
  int topbits = 2 * K - 64 * (W - 1); /* 1..64 significant bits in w[0] */
  uint64_t topmask = topbits == 64 ? ~0ull : ((1ull << topbits) - 1);
  int topshift = topbits - 2;
  for (uint64_t r = r_lo; r < r_hi; r++) {
    uint64_t b0 = off[r], b1 = off[r + 1];
    if (b1 - b0 < (uint64_t)K) continue;
    uint64_t fw[MAXW] = {0, 0, 0, 0}, rc[MAXW] = {0, 0, 0, 0};
    uint64_t filled = 0;
    for (uint64_t q = b0; q < b1; q++) {
      uint32_t b = get_base(packed, q);
      roll_fw(fw, W, topmask, b);
      roll_rc(rc, W, topshift, b);
      if (++filled >= (uint64_t)K) emit(ctx, cmp_w(fw, rc, W) <= 0 ? fw : rc);
    }
  }
}

/* bucket id = top `bbits` bits of the 2K-bit k-mer */
static inline uint32_t bucket_of(const uint64_t* k, int K, int W, int bbits) {
  int topbits = 2 * K - 64 * (W - 1);
  if (bbits == 0) return 0;
  if (topbits >= bbits) return (uint32_t)(k[0] >> (topbits - bbits));
  /* straddles words 0 and 1 */
  int rest = bbits - topbits;
  return (uint32_t)((k[0] << rest) | (k[1] >> (64 - rest)));
}

typedef struct { uint64_t* cnt; int K, W, bbits; } count_ctx;
static void emit_count(void* c, const uint64_t* k) {
  count_ctx* x = (count_ctx*)c;
  x->cnt[bucket_of(k, x->K, x->W, x->bbits)]++;
}
typedef struct { uint64_t* cur; uint64_t* keys; int K, W, bbits; } scat_ctx;
static void emit_scatter(void* c, const uint64_t* k) {
  scat_ctx* x = (scat_ctx*)c;
  uint64_t pos = x->cur[bucket_of(k, x->K, x->W, x->bbits)]++;
  for (int i = 0; i < x->W; i++) x->keys[pos * x->W + i] = k[i];
}

/* LSD byte radix sort of 1-word keys restricted to their low `bits` bits. */
static void radix_sort_u64(uint64_t* a, uint64_t* tmp, uint64_t n, int bits) {
  uint64_t* src = a; uint64_t* dst = tmp;
  for (int sh = 0; sh < bits; sh += 8) {
    uint64_t h[257]; memset(h, 0, sizeof h);
    for (uint64_t i = 0; i < n; i++) h[((src[i] >> sh) & 255) + 1]++;
    if (h[((src[0] >> sh) & 255) + 1] == n) continue; /* all in one bin */
    for (int i = 0; i < 256; i++) h[i + 1] += h[i];
    for (uint64_t i = 0; i < n; i++) dst[h[(src[i] >> sh) & 255]++] = src[i];
    uint64_t* t = src; src = dst; dst = t;
  }
  if (src != a) memcpy(a, src, n * 8);
}

static int g_cmpW;
static int cmp_q(const void* a, const void* b) { return cmp_w((const uint64_t*)a, (const uint64_t*)b, g_cmpW); }

void oracle_free(void* p) { free(p); }

/* Steps 3-4 of the algorithm above: keys[] grouped by bucket (bstart[nb+1], bucket = top bbits bits) are sorted
 * bucket by bucket and run-length counted.  Outputs malloc'd: sorted distinct k-mers, their counts. */
static int sort_count_buckets(uint64_t* keys, const uint64_t* bstart, uint32_t nb, int K, int W, int bbits, int T,
                              uint64_t** kmers_out, uint64_t** counts_out, uint64_t* n_distinct_out) {
  uint64_t N = bstart[nb];
  uint64_t* nd = (uint64_t*)calloc(nb + 1, 8);
  uint64_t* cnts = (uint64_t*)malloc((N ? N : 1) * 8); /* counts at the bucket's instance offset, compacted later */
  if (!nd || !cnts) return -2;
  int lowbits = 2 * K - bbits;
  g_cmpW = W;
#pragma omp parallel num_threads(T)
  {
    uint64_t* tmp = NULL; uint64_t tmpcap = 0;
#pragma omp for schedule(dynamic, 8)
    for (int64_t b = 0; b < (int64_t)nb; b++) {
      uint64_t lo = bstart[b], n = bstart[b + 1] - lo;
      if (!n) continue;
      uint64_t* a = keys + lo * W;
      if (W == 1) {
        if (n > tmpcap) { free(tmp); tmpcap = n + n / 4; tmp = (uint64_t*)malloc(tmpcap * 8); }
        radix_sort_u64(a, tmp, n, lowbits);
      } else {
        qsort(a, n, (size_t)W * 8, cmp_q);
      }
      uint64_t d = 0;
      for (uint64_t i = 0; i < n;) {
        uint64_t j = i + 1;
        while (j < n && cmp_w(a + i * W, a + j * W, W) == 0) j++;
        if (d != i) memmove(a + d * W, a + i * W, (size_t)W * 8);
        cnts[lo + d] = j - i;
        d++; i = j;
      }
      nd[b] = d;
    }
    free(tmp);
  }
  uint64_t D = 0;
  for (uint32_t b = 0; b < nb; b++) D += nd[b];
  uint64_t* ok = (uint64_t*)malloc((D ? D : 1) * W * 8);
  uint64_t* oc = (uint64_t*)malloc((D ? D : 1) * 8);
  if (!ok || !oc) return -2;
  uint64_t o = 0;
  for (uint32_t b = 0; b < nb; b++) {
    memcpy(ok + o * W, keys + bstart[b] * W, nd[b] * W * 8);
    memcpy(oc + o, cnts + bstart[b], nd[b] * 8);
    o += nd[b];
  }
  free(cnts); free(nd);
  *kmers_out = ok; *counts_out = oc; *n_distinct_out = D;
  return 0;
}

/* Count canonical k-mers.  Returns 0 on success.  Outputs are malloc'd:
 *   kmers  : n_distinct * W words, sorted ascending;  counts : n_distinct uint64.
 * n_instances_out (optional) = sum over reads of max(0, L-K+1). */
int oracle_count(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, int n_threads,
                 uint64_t** kmers_out, uint64_t** counts_out, uint64_t* n_distinct_out, uint64_t* n_instances_out) {
  if (K < 1 || K > 32 * MAXW) return -1;
  int W = (2 * K + 63) / 64;
  int bbits = 2 * K < 12 ? 2 * K : 12;
  uint32_t nb = 1u << bbits;
#ifdef _OPENMP
  if (n_threads <= 0) n_threads = omp_get_max_threads();
#else
  n_threads = 1;
#endif
  int T = n_threads;
  uint64_t* cnt = (uint64_t*)calloc((size_t)T * nb, 8);
  if (!cnt) return -2;
  /* split reads into T contiguous slices of ~equal bases */
  uint64_t* slice = (uint64_t*)malloc((T + 1) * 8);
  {
    uint64_t total = n_reads ? off[n_reads] - off[0] : 0;
    uint64_t r = 0;
    slice[0] = 0;
    for (int t = 1; t < T; t++) {
      uint64_t target = off[0] + total / T * t;
      while (r < n_reads && off[r] < target) r++;
      slice[t] = r;
    }
    slice[T] = n_reads;
  }
#pragma omp parallel num_threads(T)
  {
#ifdef _OPENMP
    int t = omp_get_thread_num();
#else
    int t = 0;
#endif
    count_ctx c = {cnt + (size_t)t * nb, K, W, bbits};
    roll_reads(packed, off, slice[t], slice[t + 1], K, W, emit_count, &c);
  }
  /* offsets: bucket-major, thread-minor */
  uint64_t* bstart = (uint64_t*)malloc((nb + 1) * 8);
  uint64_t run = 0;
  for (uint32_t b = 0; b < nb; b++) {
    bstart[b] = run;
    for (int t = 0; t < T; t++) { uint64_t v = cnt[(size_t)t * nb + b]; cnt[(size_t)t * nb + b] = run; run += v; }
  }
  bstart[nb] = run;
  uint64_t N = run;
  if (n_instances_out) *n_instances_out = N;
  uint64_t* keys = (uint64_t*)malloc((N ? N : 1) * W * 8);
  if (!keys) return -2;
#pragma omp parallel num_threads(T)
  {
#ifdef _OPENMP
    int t = omp_get_thread_num();
#else
    int t = 0;
#endif
    scat_ctx c = {cnt + (size_t)t * nb, keys, K, W, bbits};
    roll_reads(packed, off, slice[t], slice[t + 1], K, W, emit_scatter, &c);
  }
  free(cnt); free(slice);
  int rc = sort_count_buckets(keys, bstart, nb, K, W, bbits, T, kmers_out, counts_out, n_distinct_out);
  free(keys); free(bstart);
  return rc;
}

/* ------------------------------------------------------------------ sampled-partition oracle
 * SURVEY.md section 8(c) "human-scale check" (ii): the full k-mer set of a large read set cannot be held on the
 * host, so the oracle scans ALL reads but keeps only the canonical k-mer instances whose leading `pbits` bits
 * name a selected partition (sel[p] != 0, p < 2^pbits); those partitions are then counted exactly and compared
 * with the device's table for the same key ranges.
 *
 * oracle_sample_prefix: the selected instances, unsorted (malloc'd, n * W words).  Reads are off[] delimited, or
 * uniform (off == NULL: n_reads reads of read_len bases back to back).  n_windows_out = ALL windows seen.
 * oracle_sample_prefix_pos: the same instances, plus one word per instance (malloc'd, n words):
 * (q << 1) | canonical_is_reverse, q = the window's first base in the packed stream (off[] counts in it), reverse
 * when the canonical form is the reverse complement of the window (a palindrome counts as forward).  Reads are
 * split into equal slices in order and the slices concatenated in order, so the instances come ascending by q. */
static int sample_prefix_impl(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, uint32_t read_len, int K,
                              int pbits, const uint8_t* sel, int n_threads, uint64_t** keys_out, uint64_t** pos_out,
                              uint64_t* n_out, uint64_t* n_windows_out) {
  if (K < 1 || K > 32 * MAXW || pbits < 0 || pbits > 16 || pbits > 2 * K) return -1;
  int W = (2 * K + 63) / 64;
  const int want_pos = pos_out != NULL;
#ifdef _OPENMP
  if (n_threads <= 0) n_threads = omp_get_max_threads();
#else
  n_threads = 1;
#endif
  int T = n_threads;
  int topbits = 2 * K - 64 * (W - 1);
  uint64_t topmask = topbits == 64 ? ~0ull : ((1ull << topbits) - 1);
  int topshift = topbits - 2;
  uint64_t* cnt = (uint64_t*)calloc((size_t)T + 1, 8);
  uint64_t* win = (uint64_t*)calloc((size_t)T + 1, 8);
  uint64_t** bufs = (uint64_t**)calloc((size_t)T, sizeof(uint64_t*));
  uint64_t** pbufs = (uint64_t**)calloc((size_t)T, sizeof(uint64_t*));
  if (!cnt || !win || !bufs || !pbufs) return -2;
  int failed = 0;
#pragma omp parallel num_threads(T)
  {
#ifdef _OPENMP
    int t = omp_get_thread_num();
#else
    int t = 0;
#endif
    uint64_t r_lo = n_reads / T * t + (n_reads % T < (uint64_t)t ? n_reads % T : (uint64_t)t);
    uint64_t r_hi = n_reads / T * (t + 1) + (n_reads % T < (uint64_t)(t + 1) ? n_reads % T : (uint64_t)(t + 1));
    uint64_t n = 0, nw = 0, cap = 1u << 16;
    uint64_t* out = (uint64_t*)malloc(cap * (size_t)W * 8);   /* grows: the thread's selected instances */
    uint64_t* pout = want_pos ? (uint64_t*)malloc(cap * 8) : NULL;
    int bad = out == NULL || (want_pos && pout == NULL);
    for (uint64_t r = r_lo; r < r_hi && !bad; r++) {
      uint64_t b0 = off ? off[r] : r * (uint64_t)read_len, b1 = off ? off[r + 1] : b0 + read_len;
      if (b1 - b0 < (uint64_t)K) continue;
      if (n + (b1 - b0) > cap) {   /* room for every window of this read */
        cap = 2 * cap + (b1 - b0);
        uint64_t* nb = (uint64_t*)realloc(out, cap * (size_t)W * 8);
        if (!nb) { bad = 1; break; }
        out = nb;
        if (want_pos) {
          uint64_t* np_ = (uint64_t*)realloc(pout, cap * 8);
          if (!np_) { bad = 1; break; }
          pout = np_;
        }
      }
      if (W == 1) {
        uint64_t fw = 0, rc = 0, filled = 0;
        for (uint64_t q = b0; q < b1; q++) {
          uint32_t b = get_base(packed, q);
          fw = ((fw << 2) | b) & topmask;
          rc = (rc >> 2) | ((uint64_t)(3u - b) << topshift);
          if (++filled >= (uint64_t)K) {
            uint64_t c = fw < rc ? fw : rc;
            nw++;
            out[n] = c;
            if (want_pos) pout[n] = ((q + 1 - (uint64_t)K) << 1) | (uint64_t)(rc < fw);
            n += sel[pbits ? (uint32_t)(c >> (topbits - pbits)) : 0] != 0;
          }
        }
      } else {
        uint64_t fw[MAXW] = {0, 0, 0, 0}, rc[MAXW] = {0, 0, 0, 0};
        uint64_t filled = 0;
        for (uint64_t q = b0; q < b1; q++) {
          uint32_t b = get_base(packed, q);
          roll_fw(fw, W, topmask, b);
          roll_rc(rc, W, topshift, b);
          if (++filled >= (uint64_t)K) {
            int use_rc = cmp_w(rc, fw, W) < 0;
            const uint64_t* c = use_rc ? rc : fw;
            nw++;
            if (sel[bucket_of(c, K, W, pbits)]) {
              for (int i = 0; i < W; i++) out[n * W + i] = c[i];
              if (want_pos) pout[n] = ((q + 1 - (uint64_t)K) << 1) | (uint64_t)use_rc;
              n++;
            }
          }
        }
      }
    }
    if (bad) {
#pragma omp atomic write
      failed = 1;
    }
    cnt[t + 1] = n; win[t] = nw; bufs[t] = out; pbufs[t] = pout;
  }
  for (int t = 0; t < T; t++) cnt[t + 1] += cnt[t];   /* cnt[t] = first output slot of thread t */
  uint64_t* keys = failed ? NULL : (uint64_t*)malloc((cnt[T] ? cnt[T] : 1) * (size_t)W * 8);
  uint64_t* pos = failed || !want_pos ? NULL : (uint64_t*)malloc((cnt[T] ? cnt[T] : 1) * 8);
  if (want_pos && !pos && keys) { free(keys); keys = NULL; }
  uint64_t nw = 0;
  for (int t = 0; t < T; t++) {
    if (keys && bufs[t]) memcpy(keys + cnt[t] * W, bufs[t], (cnt[t + 1] - cnt[t]) * (size_t)W * 8);
    if (pos && pbufs[t]) memcpy(pos + cnt[t], pbufs[t], (cnt[t + 1] - cnt[t]) * 8);
    free(bufs[t]); free(pbufs[t]);
    nw += win[t];
  }
  uint64_t n_all = cnt[T];
  free(cnt); free(win); free(bufs); free(pbufs);
  if (!keys) return -2;
  *keys_out = keys; *n_out = n_all;
  if (want_pos) *pos_out = pos;
  if (n_windows_out) *n_windows_out = nw;
  return 0;
}

int oracle_sample_prefix(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, uint32_t read_len, int K, int pbits,
                         const uint8_t* sel, int n_threads, uint64_t** keys_out, uint64_t* n_out, uint64_t* n_windows_out) {
  return sample_prefix_impl(packed, off, n_reads, read_len, K, pbits, sel, n_threads, keys_out, NULL, n_out, n_windows_out);
}

int oracle_sample_prefix_pos(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, uint32_t read_len, int K,
                             int pbits, const uint8_t* sel, int n_threads, uint64_t** keys_out, uint64_t** pos_out,
                             uint64_t* n_out, uint64_t* n_windows_out) {
  return sample_prefix_impl(packed, off, n_reads, read_len, K, pbits, sel, n_threads, keys_out, pos_out, n_out,
                            n_windows_out);
}

/* oracle_count_keys: sort + count n canonical k-mer instances (W words each, any order; the array is consumed:
 * reordered in place is not promised, it is copied).  Outputs as oracle_count. */
int oracle_count_keys(const uint64_t* keys_in, uint64_t n, int K, int n_threads, uint64_t** kmers_out, uint64_t** counts_out,
                      uint64_t* n_distinct_out) {
  if (K < 1 || K > 32 * MAXW) return -1;
  int W = (2 * K + 63) / 64;
  int bbits = 2 * K < 16 ? 2 * K : 16;
  uint32_t nb = 1u << bbits;
#ifdef _OPENMP
  if (n_threads <= 0) n_threads = omp_get_max_threads();
#else
  n_threads = 1;
#endif
  int T = n_threads;
  uint64_t* cnt = (uint64_t*)calloc((size_t)T * nb, 8);
  uint64_t* bstart = (uint64_t*)malloc(((size_t)nb + 1) * 8);
  uint64_t* keys = (uint64_t*)malloc((n ? n : 1) * (size_t)W * 8);
  if (!cnt || !bstart || !keys) return -2;
#pragma omp parallel num_threads(T)
  {
#ifdef _OPENMP
    int t = omp_get_thread_num();
#else
    int t = 0;
#endif
    uint64_t lo = n / T * t + (n % T < (uint64_t)t ? n % T : (uint64_t)t);
    uint64_t hi = n / T * (t + 1) + (n % T < (uint64_t)(t + 1) ? n % T : (uint64_t)(t + 1));
    uint64_t* c = cnt + (size_t)t * nb;
    for (uint64_t i = lo; i < hi; i++) c[bucket_of(keys_in + i * W, K, W, bbits)]++;
  }
  uint64_t run = 0;
  for (uint32_t b = 0; b < nb; b++) {
    bstart[b] = run;
    for (int t = 0; t < T; t++) { uint64_t v = cnt[(size_t)t * nb + b]; cnt[(size_t)t * nb + b] = run; run += v; }
  }
  bstart[nb] = run;
#pragma omp parallel num_threads(T)
  {
#ifdef _OPENMP
    int t = omp_get_thread_num();
#else
    int t = 0;
#endif
    uint64_t lo = n / T * t + (n % T < (uint64_t)t ? n % T : (uint64_t)t);
    uint64_t hi = n / T * (t + 1) + (n % T < (uint64_t)(t + 1) ? n % T : (uint64_t)(t + 1));
    uint64_t* c = cnt + (size_t)t * nb;
    for (uint64_t i = lo; i < hi; i++) {
      uint64_t pos = c[bucket_of(keys_in + i * W, K, W, bbits)]++;
      for (int j = 0; j < W; j++) keys[pos * W + j] = keys_in[i * W + j];
    }
  }
  free(cnt);
  int rc = sort_count_buckets(keys, bstart, nb, K, W, bbits, T, kmers_out, counts_out, n_distinct_out);
  free(keys); free(bstart);
  return rc;
}

/* spectrum[f] = #distinct k-mers with count f; dense, length max_f + 1 (index 0 unused = 0). */
int oracle_spectrum(const uint64_t* counts, uint64_t n, uint64_t** spec_out, uint64_t* len_out) {
  uint64_t mx = 0;
  for (uint64_t i = 0; i < n; i++) if (counts[i] > mx) mx = counts[i];
  if (mx > (1ull << 31)) return -3;
  uint64_t* s = (uint64_t*)calloc(mx + 1, 8);
  if (!s) return -2;
  for (uint64_t i = 0; i < n; i++) s[counts[i]]++;
  *spec_out = s; *len_out = mx + 1;
  return 0;
}

/* Frequency-table lookup: count of each (already canonical or not) query k-mer,
 * 0 if absent.  Queries are canonicalised first when canonicalise != 0. */
static void revcomp_w(const uint64_t* x, uint64_t* out, int K, int W) {
  uint64_t fw[MAXW], rc[MAXW] = {0, 0, 0, 0};
  memcpy(fw, x, (size_t)W * 8);
  int topbits = 2 * K - 64 * (W - 1);
  int topshift = topbits - 2;
  for (int i = 0; i < K; i++) {
    /* take bases from the LAST base backwards: base = fw & 3, then fw >>= 2; rc = rc << 2 | (3-b) */
    uint32_t b = (uint32_t)(fw[W - 1] & 3);
    for (int j = W - 1; j > 0; j--) fw[j] = (fw[j] >> 2) | (fw[j - 1] << 62);
    fw[0] >>= 2;
    for (int j = 0; j < W - 1; j++) rc[j] = (rc[j] << 2) | (rc[j + 1] >> 62);
    rc[W - 1] = (rc[W - 1] << 2) | (3u - b);
  }
  (void)topshift;
  memcpy(out, rc, (size_t)W * 8);
}

void oracle_canonical(const uint64_t* x, uint64_t* out, int K) {
  int W = (2 * K + 63) / 64;
  uint64_t rc[MAXW];
  revcomp_w(x, rc, K, W);
  memcpy(out, cmp_w(x, rc, W) <= 0 ? x : rc, (size_t)W * 8);
}

void oracle_lookup(const uint64_t* kmers, const uint64_t* counts, uint64_t n_distinct, int K, const uint64_t* queries,
                   uint64_t n_q, int canonicalise, uint64_t* out) {
  int W = (2 * K + 63) / 64;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < (int64_t)n_q; i++) {
    uint64_t q[MAXW];
    if (canonicalise) oracle_canonical(queries + i * W, q, K);
    else memcpy(q, queries + i * W, (size_t)W * 8);
    uint64_t lo = 0, hi = n_distinct;
    while (lo < hi) {
      uint64_t mid = (lo + hi) / 2;
      if (cmp_w(kmers + mid * W, q, W) < 0) lo = mid + 1; else hi = mid;
    }
    out[i] = (lo < n_distinct && cmp_w(kmers + lo * W, q, W) == 0) ? counts[lo] : 0;
  }
}

/* Per-position k-mer frequencies of reads (what an error corrector asks the
 * table): out[p] for every window start p in the base stream; windows that
 * cross a read boundary (or reads shorter than K) get 0xFFFFFFFFFFFFFFFF. */
void oracle_read_freqs(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, const uint64_t* kmers,
                       const uint64_t* counts, uint64_t n_distinct, uint64_t* out) {
  int W = (2 * K + 63) / 64;
  uint64_t base0 = n_reads ? off[0] : 0;
  uint64_t total = n_reads ? off[n_reads] - off[0] : 0;
  for (uint64_t i = 0; i < total; i++) out[i] = ~0ull;
#pragma omp parallel for schedule(dynamic, 1024)
  for (int64_t r = 0; r < (int64_t)n_reads; r++) {
    uint64_t b0 = off[r], b1 = off[r + 1];
    if (b1 - b0 < (uint64_t)K) continue;
    for (uint64_t p = b0; p + K <= b1; p++) {
      uint64_t k[MAXW] = {0, 0, 0, 0};
      int topbits = 2 * K - 64 * (W - 1);
      uint64_t topmask = topbits == 64 ? ~0ull : ((1ull << topbits) - 1);
      for (int j = 0; j < K; j++) roll_fw(k, W, topmask, get_base(packed, p + j));
      uint64_t c;
      oracle_lookup(kmers, counts, n_distinct, K, k, 1, 1, &c);
      out[p - base0] = c;
    }
  }
}

/* Occurrence records: the (read id, signed position) payload of every k-mer instance, grouped by
 * canonical k-mer in table order (kmers = the sorted distinct k-mers oracle_count returned) and, inside
 * a k-mer's run, ascending by (read id, position).  pos is 1-based in the read, negative when the
 * canonical form is the reverse complement of the read's window, positive otherwise (palindromes
 * included).  run_off_out[n_distinct + 1]; read_id_out / pos_out hold one entry per instance.
 * Restates the record layout SURVEY.md section 8(a) attributes to SortKmers / KmerParcels ([U]: no
 * reference source was available -- parity unpinned).  Reads are walked in order, so each run fills
 * in (read id, position) order by construction. */
int oracle_occurrences(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, const uint64_t* kmers,
                       uint64_t n_distinct, uint64_t* run_off_out, uint32_t* read_id_out, int32_t* pos_out) {
  if (K < 1 || K > 32 * MAXW) return -1;
  int W = (2 * K + 63) / 64;
  int topbits = 2 * K - 64 * (W - 1);
  uint64_t topmask = topbits == 64 ? ~0ull : ((1ull << topbits) - 1);
  int topshift = topbits - 2;
  uint64_t* cur = (uint64_t*)calloc(n_distinct + 1, 8);
  if (!cur) return -2;
  for (int pass = 0; pass < 2; pass++) {
    for (uint64_t r = 0; r < n_reads; r++) {
      uint64_t b0 = off[r], b1 = off[r + 1];
      if (b1 - b0 < (uint64_t)K) continue;
      uint64_t fw[MAXW] = {0, 0, 0, 0}, rc[MAXW] = {0, 0, 0, 0};
      for (uint64_t q = b0; q < b1; q++) {
        uint32_t b = get_base(packed, q);
        roll_fw(fw, W, topmask, b);
        roll_rc(rc, W, topshift, b);
        if (q - b0 + 1 < (uint64_t)K) continue;
        int use_rc = cmp_w(rc, fw, W) < 0;
        const uint64_t* c = use_rc ? rc : fw;
        uint64_t lo = 0, hi = n_distinct;
        while (lo < hi) {
          uint64_t mid = (lo + hi) / 2;
          if (cmp_w(kmers + mid * W, c, W) < 0) lo = mid + 1; else hi = mid;
        }
        if (lo >= n_distinct || cmp_w(kmers + lo * W, c, W) != 0) { free(cur); return -3; }
        if (pass == 0) {
          cur[lo]++;
        } else {
          uint64_t slot = cur[lo]++;
          int32_t p1 = (int32_t)(q - b0 + 1 - (uint64_t)K) + 1;
          read_id_out[slot] = (uint32_t)r;
          pos_out[slot] = use_rc ? -p1 : p1;
        }
      }
    }
    if (pass == 0) {
      uint64_t run = 0;
      for (uint64_t i = 0; i < n_distinct; i++) { uint64_t v = cur[i]; run_off_out[i] = run; cur[i] = run; run += v; }
      run_off_out[n_distinct] = run;
    }
  }
  free(cur);
  return 0;
}

int oracle_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
