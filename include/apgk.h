/*
 * apgk.h -- C ABI of libapgk.so, the B200-native k-mer spectrum engine that
 * replaces ALLPATHS-LG's k-mer hot path (extract -> canonicalise -> sort ->
 * count -> spectrum, plus the frequency-table lookups error correction makes).
 *
 * REFERENCE INTERFACES REPLACED.  The reference tree was not available when
 * this was written (/root/reference held one empty README; SURVEY.md section 0),
 * so the entry points below cite the reference by the names BASELINE.json's
 * north_star gives them, with the unverified locations SURVEY.md section 2.2 / A.1
 * recalls.  No file:line exists to cite; each is marked [BJ] (named by
 * BASELINE.json) or [U] (unverified recollection).
 *
 *   apgk_add_reads*      <- the vecbasevector& argument of the builders
 *                           (src/Basevector.h, src/feudal/BaseVec.h [U])
 *   apgk_finish          <- SortKmers<K,...>(...) and KmerParcelsBuilder::Build()
 *                           (src/kmers/SortKmers.{h,cc},
 *                            src/kmers/kmer_parcels/KmerParcelsBuilder.{h,cc} [BJ names, U paths]);
 *                           naif_kmerize(kernel, n_threads) (src/kmers/naif_kmer/ [U])
 *   apgk_spectrum*       <- class KmerSpectrum (src/kmers/KmerSpectra.h [BJ name, U path])
 *   apgk_counts_*        <- the sorted (k-mer, frequency) records: vec<kmer_record>,
 *                           KmerParcelReader batches, KmerKmerFreq vectors [U]
 *   apgk_*occurrences*   <- the (read id, signed position) payload of SortKmers' kmer records and
 *                           KmerParcels' batches (src/kmers/KmerRecord.h, kmer_parcels/ [U])
 *   apgk_lookup*, apgk_read_freqs*
 *                        <- the k-mer frequency tables FindErrors queries per read
 *                           position (src/paths/FindErrors*.cc [BJ name, U path])
 *
 * CONVENTIONS (SURVEY.md section 8 "Definition"): bases A=0 C=1 G=2 T=3, packed
 * 2 bits per base, base q of a buffer at bits [2q, 2q+2) (little-endian inside
 * a byte).  A k-mer is the 2K-bit integer with its first base most significant,
 * stored in W = ceil(2K/64) uint64 words, most significant word first, value
 * right-aligned.  canonical(x) = min(x, revcomp(x)).  count = number of window
 * instances with that canonical form.  spectrum[f] = number of distinct
 * canonical k-mers with count f.
 *
 * Every function returns APGK_OK (0) or a negative error code and never
 * aborts or throws; apgk_last_error() describes the last failure.  There is no
 * CPU fallback: without a CUDA device apgk_create fails with APGK_E_CUDA.
 * A context is single-caller.  Inputs are borrowed for the duration of a call;
 * outputs are library-owned until apgk_reset / apgk_destroy.
 */
#ifndef APGK_H
#define APGK_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APGK_OK 0
#define APGK_E_ARG (-1)      /* bad argument */
#define APGK_E_CUDA (-2)     /* CUDA runtime error / no device */
#define APGK_E_NOMEM (-3)    /* device or host allocation failed */
#define APGK_E_STATE (-4)    /* call out of order (e.g. results before apgk_finish) */
#define APGK_E_RANGE (-5)    /* a size exceeds what this build handles (see message) */

#define APGK_WANT_SPECTRUM 1u /* always produced */
#define APGK_WANT_COUNTS 2u   /* also build the sorted (k-mer, count) table + lookup index */
/* Streamed ingest: apgk_add_reads_uniform (byte-aligned appends) returns before its host-to-device copy
 * has completed.  `packed` must then stay valid -- and should be pinned (apgk_host_alloc) -- until the
 * next apgk_finish / apgk_partition has returned; that call runs its level-0 histogram slice by slice
 * behind the copy instead of after it.  Every other call waits for the copy first. */
#define APGK_ASYNC_INGEST 4u

#define APGK_MAX_K 96

typedef struct apgk_ctx apgk_ctx;

typedef struct {
  int32_t K;            /* 1..APGK_MAX_K */
  int32_t device;       /* CUDA device ordinal */
  uint32_t flags;       /* APGK_WANT_* */
  int32_t prefix_bits;  /* 0 = auto; else total bits of the two partition levels (2..24) */
  uint64_t reserve_bases; /* 0 or a hint: pre-size the device read store for this many bases */
  uint64_t max_round_keys; /* 0 = auto (from free device memory); else the most k-mer instances one
                              k-mer-space round may hold -- more rounds, less memory */
  uint64_t max_inner_keys; /* 0 = auto.  Rounds have two levels: an OUTER round extracts the k-mers of a range
                              of leading-bit buckets once (8*W bytes per instance), its INNER rounds run the
                              second partition level and the counting over sub-ranges (4 or 8*W, + 4 bytes per
                              instance).  max_round_keys bounds the outer rounds, this field the inner ones
                              (default: max_round_keys when that is set) */
} apgk_config;

/* Parameters of the synthetic read generator (SURVEY.md section 8d); identical in the oracle. */
typedef struct {
  uint64_t genome_len;
  uint64_t seed_g, seed_p, seed_q, seed_r, seed_e;
  uint32_t read_len;
  uint32_t err_per_200; /* 1 = 0.5 % substitutions, 0 = none */
} apgk_synth_params;

int apgk_create(const apgk_config* cfg, apgk_ctx** out);
void apgk_destroy(apgk_ctx* ctx);
const char* apgk_last_error(const apgk_ctx* ctx);
int apgk_words_per_kmer(int K);

/* Drop reads and results, keep device buffers (for reuse in a streaming loop). */
int apgk_reset(apgk_ctx* ctx);

/* ---- reads in.  May be called repeatedly; reads accumulate in the device store.
 * packed/off are HOST buffers: read r = bases off[r] .. off[r+1]-1 of `packed`. */
int apgk_add_reads(apgk_ctx* ctx, const uint8_t* packed, const uint64_t* off, uint64_t n_reads);
/* n_reads reads of read_len bases each, back to back, starting at base first_base of `packed`. */
int apgk_add_reads_uniform(apgk_ctx* ctx, const uint8_t* packed, uint64_t first_base, uint64_t n_reads,
                           uint32_t read_len);
/* Generate synthetic reads [r0, r0+n) straight into the device store (store must be empty or
 * hold a multiple of 16 bases). */
int apgk_synth_reads(apgk_ctx* ctx, const apgk_synth_params* p, uint64_t r0, uint64_t n_reads);
/* Copy the device store's packed bases to a host buffer of ceil(total_bases/32)*8 bytes. */
int apgk_export_reads(apgk_ctx* ctx, uint8_t* packed_out);
int apgk_read_store_info(const apgk_ctx* ctx, uint64_t* total_bases, uint64_t* n_reads);

/* ---- the hot path: extract + canonicalise + partition + sort + count + spectrum. */
int apgk_finish(apgk_ctx* ctx);

/* ---- results */
int apgk_totals(const apgk_ctx* ctx, uint64_t* n_instances, uint64_t* n_distinct);
/* Dense spectrum: (*spec)[f] for f in [0, *len); (*spec)[0] == 0.  APGK_E_RANGE if the largest
 * count would need more than 2^28 entries -- use apgk_spectrum_sparse then. */
int apgk_spectrum(apgk_ctx* ctx, const uint64_t** spec, uint64_t* len);
/* Sparse spectrum: *n pairs (freq[i], n_kmers[i]) with n_kmers > 0, ascending freq. */
int apgk_spectrum_sparse(apgk_ctx* ctx, const uint64_t** freq, const uint64_t** n_kmers, uint64_t* n);
/* Sorted table on the DEVICE: kmers = n_distinct * W words, counts = n_distinct uint32
 * (saturating at 0xFFFFFFFF).  Needs APGK_WANT_COUNTS. */
int apgk_counts_device(apgk_ctx* ctx, const uint64_t** d_kmers, const uint32_t** d_counts, uint64_t* n_distinct);
/* Copy records [first, first+n) of the table to host buffers (either may be NULL). */
int apgk_counts_copy(apgk_ctx* ctx, uint64_t first, uint64_t n, uint64_t* kmers_out, uint32_t* counts_out);

/* Give the scratch buffers of the pipeline back to the device (the k-mers of the partition levels, temp records,
 * occurrence records): the read store, the result table with its index and the spectrum stay, so lookups keep
 * working; the next count allocates again. */
int apgk_release_temp(apgk_ctx* ctx);
/* Sizing hint, before a count: room for n_records (k-mer, count) records, so that a table that grows round by
 * round is never reallocated (a reallocation copies it and needs both copies for a moment).  Discards a
 * smaller table. */
int apgk_reserve_table(apgk_ctx* ctx, uint64_t n_records);
/* Records [*first, *first + *n) of the sorted table are exactly the k-mers whose leading prefix_bits bits equal
 * `prefix` (one parcel of k-mer space; read off the table's prefix index).  prefix_bits <= D0 + D1 of
 * apgk_geometry.  On a shard context only the k-mers the shard owns are there. */
int apgk_prefix_range(apgk_ctx* ctx, int32_t prefix_bits, uint64_t prefix, uint64_t* first, uint64_t* n);

/* ---- frequency-table queries (need APGK_WANT_COUNTS and a finished context) */
/* counts_out[i] = count of query k-mer i (W words each, host), 0 if absent.  Queries are
 * canonicalised first when canonicalise != 0. */
int apgk_lookup(apgk_ctx* ctx, const uint64_t* kmers, uint64_t n, int canonicalise, uint32_t* counts_out);
/* out[i] = count of the canonical k-mer starting at base first_base+i of the device read store,
 * 0xFFFFFFFF where the window crosses a read end.  out is a HOST buffer of n_bases entries. */
int apgk_read_freqs(apgk_ctx* ctx, uint64_t first_base, uint64_t n_bases, uint32_t* out);
/* The same for EVERY base of the store into a DEVICE buffer of total_bases entries (what an error
 * corrector that keeps the reads on the GPU asks).  Bulk form: one sweep sends every window to its
 * prefix bucket, one CTA per bucket resolves the bucket's windows against its keys in shared memory
 * (the context's table must have been counted from its own read store by apgk_finish).  apgk_read_freqs
 * over the whole store takes this path too.  ms3 (may be NULL) = device milliseconds of {clear + run
 * offsets, sweep, per-bucket resolution}. */
int apgk_read_freqs_device(apgk_ctx* ctx, uint32_t* d_out, float* ms3);

/* ---- k-mer occurrence records: the payload half of the reference's SortKmers records (k-mer, read id,
 * signed position) and KmerParcels batches (k-mer + list of (read id, position)) [BJ names, U layout;
 * SURVEY.md section 8(a) rows 1-2, 8(f) rank 2].  Needs a context finished by apgk_finish with
 * APGK_WANT_COUNTS whose read store is still in place.  For distinct k-mer i of the sorted table, its
 * count[i] instances occupy slots [run_off[i], run_off[i+1]) of the occurrence list, ascending by
 * (read id, position); run_off[n_distinct] == n_instances.  Read ids number the reads in the order they
 * were added (reads without bases included).  pos is 1-based within the read and NEGATIVE when the
 * canonical form is the reverse complement of the read's window (a palindrome counts as forward). */
int apgk_build_occurrences(apgk_ctx* ctx);
/* n_occ = n_instances; n_big_runs = runs sorted by the CTA-wide network (> 256 instances);
 * ms5 = device milliseconds of {run-offset scan, sweep of the reads (scatter to buckets), per-bucket
 * placement, per-run sort, big-run sort}. */
int apgk_occurrences_info(const apgk_ctx* ctx, uint64_t* n_occ, uint64_t* n_big_runs, float* ms5);
/* DEVICE pointers, library-owned until the next finish / reset: run offsets (uint64[n_distinct+1]) and
 * the occurrences encoded as (global base position in the read store << 1) | canonical_is_reverse. */
int apgk_occurrences_device(apgk_ctx* ctx, const uint64_t** d_run_off, const uint64_t** d_occ, uint64_t* n_occ);
/* HOST copies for k-mers [first_kmer, first_kmer + n_kmers): run_off_out[n_kmers+1] (absolute slots; may
 * be NULL), and read_id_out / pos_out for slots [run_off[first_kmer], run_off[first_kmer+n_kmers)) (both
 * NULL = offsets only, to size the buffers). */
int apgk_occurrences_copy(apgk_ctx* ctx, uint64_t first_kmer, uint64_t n_kmers, uint64_t* run_off_out,
                          uint32_t* read_id_out, int32_t* pos_out);

/* ---- multi-GPU building blocks (one context per rank; the exchange itself is the caller's,
 * e.g. NCCL all-to-all).  Canonical k-mers are owned by rank hash(kmer) % n_ranks. */
/* Pass 1: per-owner instance counts of this rank's reads (counts_out[n_ranks], host). */
int apgk_owner_plan(apgk_ctx* ctx, uint32_t n_ranks, uint64_t* counts_out);
/* Pass 2: write this rank's canonical k-mers grouped by owner (owner 0 first) into the DEVICE
 * buffer d_keys_out (sum(counts) * W words). */
int apgk_owner_scatter(apgk_ctx* ctx, uint64_t* d_keys_out);
/* The library's own level-0 key buffer, sized for n_keys k-mers: a caller may use it as the
 * d_keys_out of apgk_owner_scatter (and as the SEND buffer of its exchange) instead of allocating
 * another N*W words.  Its contents are overwritten by the next apgk_finish* call -- so it cannot be the
 * d_keys of apgk_finish_keys_device (refused with APGK_E_ARG): receive into a buffer of your own. */
int apgk_key_buffer(apgk_ctx* ctx, uint64_t n_keys, uint64_t** d_ptr);
/* Owner hash of k-mers (host arrays), for tests. */
int apgk_owner_of(int K, const uint64_t* kmers, uint64_t n, uint32_t n_ranks, uint32_t* owner_out);
/* Sort + count a DEVICE array of n canonical k-mers (W words each) instead of the read store. */
int apgk_finish_keys_device(apgk_ctx* ctx, const uint64_t* d_keys, uint64_t n);
/* Device pointer to the dense spectrum accumulator (uint64[65536]) after finish, for all-reduce;
 * apgk_spectrum_reload() re-reads it after the caller summed it in place. */
int apgk_spectrum_device(apgk_ctx* ctx, uint64_t** d_spec, uint64_t* len);
int apgk_spectrum_reload(apgk_ctx* ctx);

/* ---- multi-GPU, partition-first form (the one allpathslg_b200.dist.sharded_count uses): every rank
 * partitions ITS reads by the leading prefix_bits of the canonical k-mer (levels 0 and 1 of the
 * single-GPU pipeline, nothing else), the ranks agree on balanced bucket ranges from the summed
 * bucket histogram, exchange whole bucket ranges of level-1 elements (32-bit remainders when they
 * fit) and each rank sorts + counts the ranges it owns.  A k-mer's owner is a function of the
 * canonical k-mer alone, so counts are final without a merge; compared with the hash form above
 * the k-mers are extracted and partitioned once, not twice, and half the bytes cross NVLink. */
/* Upper bound of the k-mer instances in the read store (what the geometry choice is based on). */
int apgk_window_upper(const apgk_ctx* ctx, uint64_t* upper);
/* Prefix bits a run over `upper` instances would pick.  Ranks call it with the maximum over ranks
 * and pass the result to apgk_partition so that all of them use the same geometry. */
int apgk_choose_prefix_bits(apgk_ctx* ctx, uint64_t upper, int32_t* prefix_bits);
/* Levels 0+1 over the read store with 2^prefix_bits buckets (0 = choose).  APGK_E_RANGE when the
 * k-mers would need more than one k-mer-space round on this device: run the rounds with
 * apgk_level0_totals + apgk_partition_range then. */
int apgk_partition(apgk_ctx* ctx, int32_t prefix_bits);
/* K-mer-space rounds of the sharded form (a rank whose k-mers do not fit one round): the same two levels
 * restricted to the level-0 buckets [d0_lo, d0_hi) -- the leading D0 bits of the canonical k-mer, D0 as
 * apgk_geometry reports it for this prefix_bits.  Buckets outside the range come out empty.  The caller runs
 * the rounds: partition_range -> exchange -> apgk_count_pieces* -> harvest the round's spectrum / table ->
 * next range (allpathslg_b200.dist does, with the same ranges on every rank). */
int apgk_partition_range(apgk_ctx* ctx, int32_t prefix_bits, int32_t d0_lo, int32_t d0_hi);
/* Level-0 bucket totals (k-mer instances per leading-D0-bits bucket, HOST, *n_level0 = 2^D0 entries) of the last
 * apgk_partition* call on this context -- also after one that failed with APGK_E_RANGE -- and the number of
 * instances one round may hold under the device-memory budget; what the ranks need to agree on the ranges. */
int apgk_level0_totals(apgk_ctx* ctx, uint64_t* totals_out, uint32_t cap, uint32_t* n_level0, uint64_t* round_capacity);
/* Result of apgk_partition, all DEVICE pointers owned by the library: bucket sizes
 * (uint64[n_buckets]), the elements grouped by bucket (elem_bytes each: 4, or 8 * W). */
int apgk_partition_info(apgk_ctx* ctx, const uint64_t** d_bucket_sizes, uint64_t* n_buckets, void** d_elems,
                        uint32_t* elem_bytes, uint64_t* n_elems);
/* Receiver side.  d_recv (DEVICE) holds n_src segments, segment s starting at element seg_off[s]
 * (HOST array) and containing source s's pieces of buckets [bucket_lo, bucket_hi) in bucket order;
 * d_sizes_all (DEVICE, uint32[n_src][n_buckets]) are the piece sizes.  A merged bucket holds the
 * instances of all the sources, so each is first cut into 2^split_bits sub-buckets by its next
 * remainder bits (pass ceil(log2(n_src)); clamped by the library).  Sorts + counts the shard:
 * afterwards the context answers totals / spectrum / counts / lookups for the k-mers it owns. */
int apgk_count_pieces(apgk_ctx* ctx, const void* d_recv, uint32_t n_src, const uint32_t* d_sizes_all,
                      const uint64_t* seg_off, uint64_t bucket_lo, uint64_t bucket_hi, int32_t split_bits);

/* Same, with the exchange fused into the gather: d_src_base[s] (HOST array of DEVICE pointers) is
 * source s's partition buffer -- its own for s == this rank (NULL selects it), a peer's buffer mapped
 * with apgk_peer_open otherwise -- and src_off[s] the element offset of bucket_lo's piece in it.  The
 * gather kernel then reads the pieces straight over NVLink peer memory: no all-to-all, no receive
 * buffer, the transfer overlaps the splitting.  The peers must not touch their partition buffers
 * until every rank has returned from this call (the spectrum all-reduce that follows is that barrier).
 * d_sub_sizes (DEVICE, uint32[n_src][(bucket_hi - bucket_lo) << bits], may be NULL) are the senders'
 * own sub-bucket counts (apgk_partition_subsizes) for this range: with them the pieces cross NVLink
 * once instead of twice. */
int apgk_count_pieces_peer(apgk_ctx* ctx, const void* const* d_src_base, uint32_t n_src, const uint32_t* d_sizes_all,
                           const uint64_t* src_off, uint64_t bucket_lo, uint64_t bucket_hi, int32_t split_bits,
                           const uint32_t* d_sub_sizes);
/* Sender side of that: sizes of the 2^bits sub-buckets of every bucket of this context's partition
 * (DEVICE, uint32[n_buckets << bits], library-owned); *effective_bits is the clamped split_bits. */
int apgk_partition_subsizes(apgk_ctx* ctx, int32_t split_bits, int32_t* effective_bits, const uint32_t** d_sub_sizes);
/* CUDA IPC plumbing for the peer form: export this context's partition buffer (64-byte handle, valid
 * until the buffer is reallocated by a larger run), map a peer's handle, unmap it. */
int apgk_partition_export(apgk_ctx* ctx, uint8_t handle_out[64]);
int apgk_peer_open(apgk_ctx* ctx, const uint8_t handle[64], void** d_ptr);
int apgk_peer_close(apgk_ctx* ctx, void* d_ptr);

/* ---- sharded counting behind the C ABI: a GROUP of ranks, one context (one GPU) each.
 * This is SURVEY.md section 8(e) / BASELINE.json's "k-mers are partitioned by canonical k-mer ... each rank sorts and
 * counts its own shard, and the per-rank spectra are summed" as ONE call: apgk_group_count runs, on every rank,
 * levels 0 + 1 over the rank's read store, the all-gather of the bucket histograms, the balanced bucket ranges, the
 * exchange fused into the gather kernel over NVLink peer memory, the per-bucket counting of the owned range and
 * the spectrum all-reduce -- in k-mer-space rounds when a rank's k-mers do not fit its device at once (every
 * round's shard table is appended, so each context ends up with the table of ALL the k-mers it owns).
 * Two ways to form a group:
 *   multi-process (one process per GPU, e.g. under mpirun / torchrun): rank 0 calls apgk_group_unique_id, the host
 *     program hands the 128 bytes to every rank by its own means, every rank calls apgk_group_join.  The small
 *     collectives use NCCL (libnccl.so.2 is loaded on first use); the partition buffers are mapped with CUDA IPC.
 *   single process (one host thread drives all GPUs, as an ALLPATHS-LG module would): apgk_group_local over
 *     contexts created on different devices (or, for tests, on one device); no NCCL is involved.
 * All group calls are collective: every rank (every process of the multi-process form) must make them in the
 * same order.  A group borrows its contexts: destroy the group first. */
typedef struct apgk_group apgk_group;
#define APGK_GROUP_ID_BYTES 128
int apgk_group_unique_id(uint8_t id_out[APGK_GROUP_ID_BYTES]);
int apgk_group_join(apgk_ctx* ctx, const uint8_t id[APGK_GROUP_ID_BYTES], int32_t rank, int32_t world, apgk_group** out);
int apgk_group_local(apgk_ctx* const* ctxs, int32_t n, apgk_group** out);
void apgk_group_destroy(apgk_group* g);
const char* apgk_group_last_error(const apgk_group* g);
/* The sharded hot path over the read stores the group's contexts hold now.  Afterwards every context answers
 * apgk_totals / apgk_counts_* / apgk_lookup / apgk_prefix_range for the k-mers it owns, and the group the
 * global results below (identical on every rank). */
int apgk_group_count(apgk_group* g);
int apgk_group_totals(const apgk_group* g, uint64_t* n_instances, uint64_t* n_distinct);
/* Global spectrum, sparse form as apgk_spectrum_sparse (library-owned until the next apgk_group_count). */
int apgk_group_spectrum_sparse(apgk_group* g, const uint64_t** freq, const uint64_t** n_kmers, uint64_t* n);
typedef struct {
  int32_t world, n_rounds, n_outer_rounds, prefix_bits, split_bits, peer_exchange; /* peer_exchange: 1 = gather over peer memory */
  uint64_t shard_instances;   /* k-mer instances this rank (the group's first local context) counted */
  uint64_t remote_bytes;      /* bytes its gather kernels read from the peers (NVLink) */
  float gather_ms;            /* device time of those kernels */
  float step_ms;              /* device time of the whole call on that context's stream */
} apgk_group_stats;
int apgk_group_stats_get(const apgk_group* g, apgk_group_stats* out);
/* Frequency lookups on the sharded table: the bulk form of apgk_read_freqs for a group.  Each rank's reads contain
 * k-mers every rank owns, so the queries travel to their owner: per batch of the base range, every rank sends its
 * windows' level-1 elements (4-byte remainder or full key) bucket by bucket through its partition buffer, each owner
 * resolves the pieces of the buckets it owns against its table over peer memory and writes the counts back in place,
 * and every rank scatters the answers to the positions.  Batches are sized from the device-memory budget of the
 * count; every rank runs the same number of them.
 * After apgk_group_count with APGK_WANT_COUNTS: for every base i of [first_base[j], first_base[j] + n_bases[j]) of the
 * read store of the group's j-th LOCAL context, d_out[j][i - first_base[j]] = the GLOBAL count of the canonical k-mer
 * starting there (0xFFFFFFFF where the window leaves its read).  This is what apgk_read_freqs_device gives on one GPU,
 * with the counts held by the shards.  Collective.  Arrays have one entry per local context (one in the multi-process
 * form).  d_out: DEVICE buffers of n_bases[j] uint32 on that context's device (NULL allowed where n_bases[j] == 0).
 * stats may be NULL.  Errors are decided from values all ranks share and come back identical on every rank:
 * APGK_E_STATE without a current count with APGK_WANT_COUNTS, or when a member context was reset, given reads or
 * counted on its own since (apgk_release_temp is fine), or when a window's k-mer is missing from its owner's table;
 * APGK_E_ARG for a range beyond a read store or a missing buffer; APGK_E_NOMEM when a rank's buffers do not fit. */
typedef struct {
  int32_t n_batches;        /* exchange batches this call ran (agreed by all ranks) */
  uint64_t n_queries;       /* valid windows of this rank's range that were resolved */
  uint64_t remote_bytes;    /* bytes this rank's owner-side kernels read from and wrote to peers' memory */
  float sweep_ms, exchange_ms, scatter_ms, total_ms;   /* device time, first local context */
} apgk_group_freq_stats;
int apgk_group_read_freqs_device(apgk_group* g, uint32_t* const* d_out, const uint64_t* first_base,
                                 const uint64_t* n_bases, apgk_group_freq_stats* stats);

/* ---- instrumentation */
#define APGK_N_STAGES 14
/* Device milliseconds of the last finish, by stage; names via apgk_stage_name(i). */
int apgk_stage_ms(const apgk_ctx* ctx, float* ms_out /* [APGK_N_STAGES] */);
const char* apgk_stage_name(int i);
/* Number of kernels this library launched since creation (or the last apgk_reset_counters). */
uint64_t apgk_kernel_launches(const apgk_ctx* ctx);
void apgk_reset_counters(apgk_ctx* ctx);
/* Geometry of the last finish: D0, D1, REM bits, element bytes of the level-1 buffer, number of
 * oversize buckets (k_big), number of buckets deferred to the general kernel, bucket capacity,
 * number of k-mer-space rounds. */
int apgk_geometry(const apgk_ctx* ctx, int32_t* out8);
/* Device buffers for callers without their own allocator (e.g. the exchange buffers of the
 * multi-GPU path in a plain C++ host), and a synchronous device-to-host copy. */
int apgk_device_alloc(apgk_ctx* ctx, void** p, size_t bytes);
int apgk_device_free(apgk_ctx* ctx, void* p);
int apgk_device_copy_to_host(apgk_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes);
/* Pinned host memory helpers for callers that stream batches. */
int apgk_host_alloc(void** p, size_t bytes);
int apgk_host_free(void* p);

/* Diagnostics of the full-key per-bucket kernel since the last reset: out8[0] passes, [1] passes that
 * overflowed a row (range split), [2] passes redone for a tag collision, [3] buckets. */
int apgk_debug_counters(apgk_ctx* ctx, uint64_t* out8, int reset);
/* ---- test hooks: run the device code's inline helpers on the HOST (no GPU needed).  They exist
 * so the CPU test-suite can check extraction against the oracle; the library never calls them. */
int apgk_debug_host_extract(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K,
                            uint64_t* kmers_out /* total_bases * W */, uint8_t* valid_out /* total_bases */);
int apgk_debug_host_canonical(int K, const uint64_t* kmers, uint64_t n, uint64_t* out);
/* level-0 digit (top D bits of the canonical k-mer) of every window start, via the cheap top-bits identity */
int apgk_debug_host_topdigits(const uint8_t* packed, const uint64_t* off, uint64_t n_reads, int K, int D,
                              uint32_t* digits_out /* total_bases */);
/* table_find_index (the interpolated search of the lookups) on the HOST over a sorted key array with a
 * prefix index of prefix_bits bits built here; idx_out[i] = index of query i or UINT64_MAX. */
int apgk_debug_host_table_find(int K, const uint64_t* sorted_kmers, uint64_t n, int prefix_bits, const uint64_t* queries,
                               uint64_t n_q, uint64_t* idx_out);
int apgk_debug_host_synth(const apgk_synth_params* p, uint64_t r0, uint64_t n_reads, uint8_t* packed_out);
/* The sharded form's ownership rule on the HOST: bounds_out[world + 1] = the contiguous bucket ranges of equal cost
 * (cost of a non-empty bucket = its size + bucket_cost; bucket_cost 0 = equal instance counts) that the device's
 * k_total_sizes -> scan -> k_splitters derive from the all-gathered bucket sizes. */
int apgk_debug_host_splitters(const uint32_t* bucket_sizes, uint32_t n_buckets, uint32_t world, uint32_t bucket_cost,
                              uint32_t* bounds_out);

#ifdef __cplusplus
}
#endif
#endif /* APGK_H */
