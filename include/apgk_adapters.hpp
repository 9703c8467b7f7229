// apgk_adapters.hpp -- header-only C++ host layer over the C ABI (include/apgk.h).
//
// The reference is a C++ code base, so its k-mer layer would sit on libapgk.so
// through classes with the reference's own names.  The reference tree was not
// available (SURVEY.md section 0): names follow BASELINE.json's north_star
// (SortKmers, KmerParcelsBuilder, KmerSpectrum, the FindErrors frequency
// tables) and SURVEY.md's unverified recollection of their shape -- builders
// constructed from (K, reads, n_threads) with a Build() call, a spectrum that
// IS a vector indexed by frequency with text I/O, errors that abort.  Here a
// failed C call throws std::runtime_error carrying apgk_last_error().
//
// Nothing in this file computes k-mers on the CPU: every result comes from the
// CUDA library.  Link with -lapgk.
#pragma once
#include <cstdint>
#include <cstdio>
#include <fstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "apgk.h"

namespace apgk_ref {

// Minimal stand-in for the reference's vecbasevector: 2-bit packed reads + base offsets,
// exactly the buffers apgk_add_reads takes.
class vecbasevector {
 public:
  vecbasevector() : off_(1, 0) {}
  void push_back(const std::string& acgt) {
    const uint64_t q0 = off_.back();
    packed_.resize(((q0 + acgt.size() + 31) / 32) * 8 + 8, 0);
    for (size_t j = 0; j < acgt.size(); j++) {
      const uint64_t q = q0 + j;
      packed_[q >> 2] |= (uint8_t)(code(acgt[j]) << ((q & 3) * 2));
    }
    off_.push_back(q0 + acgt.size());
  }
  size_t size() const { return off_.size() - 1; }
  uint64_t read_len(size_t i) const { return off_[i + 1] - off_[i]; }
  const uint8_t* packed() const { return packed_.data(); }
  const uint64_t* offsets() const { return off_.data(); }

 private:
  static unsigned code(char c) {
    switch (c) {
      case 'A': case 'a': return 0;
      case 'C': case 'c': return 1;
      case 'G': case 'g': return 2;
      case 'T': case 't': return 3;
    }
    throw std::invalid_argument("vecbasevector: only ACGT can be packed");
  }
  std::vector<uint8_t> packed_;
  std::vector<uint64_t> off_;
};

// RAII engine context.
class Engine {
 public:
  Engine(int K, bool want_counts, int device = 0) : K_(K), W_(apgk_words_per_kmer(K)) {
    apgk_config cfg{};
    cfg.K = K; cfg.device = device; cfg.flags = APGK_WANT_SPECTRUM | (want_counts ? APGK_WANT_COUNTS : 0);
    const int rc = apgk_create(&cfg, &ctx_);
    if (rc != APGK_OK)
      throw std::runtime_error("apgk_create failed (rc " + std::to_string(rc) + "): no CUDA device? there is no CPU fallback");
  }
  ~Engine() { apgk_destroy(ctx_); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;
  void ck(int rc) const {
    if (rc != APGK_OK) throw std::runtime_error(std::string("apgk: ") + apgk_last_error(ctx_));
  }
  void AddReads(const vecbasevector& r) { ck(apgk_add_reads(ctx_, r.packed(), r.offsets(), r.size())); }
  void Finish() { ck(apgk_finish(ctx_)); }
  apgk_ctx* ctx() const { return ctx_; }
  int K() const { return K_; }
  int W() const { return W_; }

 private:
  apgk_ctx* ctx_ = nullptr;
  int K_, W_;
};

// `class KmerSpectrum`: a vector indexed by k-mer frequency.
class KmerSpectrum : public std::vector<uint64_t> {
 public:
  explicit KmerSpectrum(int K) : K_(K) {}
  int K() const { return K_; }
  void FromReads(const vecbasevector& reads, int device = 0) {
    Engine e(K_, /*want_counts=*/false, device);
    e.AddReads(reads);
    e.Finish();
    FromEngine(e);
  }
  void FromEngine(const Engine& e) {
    const uint64_t* s = nullptr; uint64_t n = 0;
    e.ck(apgk_spectrum(e.ctx(), &s, &n));
    assign(s, s + n);
  }
  uint64_t NumDistinct() const { uint64_t t = 0; for (uint64_t v : *this) t += v; return t; }
  uint64_t NumInstances() const { uint64_t t = 0; for (size_t f = 0; f < size(); f++) t += f * (*this)[f]; return t; }
  void Write(const std::string& path) const {
    std::ofstream o(path);
    o << "# kmer spectrum K=" << K_ << "\n";
    for (size_t f = 0; f < size(); f++) if ((*this)[f]) o << f << " " << (*this)[f] << "\n";
  }

 private:
  int K_;
};

// One record of the sorted table: W words (most significant first) and the multiplicity.
template <int W>
struct kmer_count {
  uint64_t kmer[W];
  uint32_t count;
};

// `SortKmers`: all canonical k-mers of the reads, ascending, with counts.
template <int K>
void SortKmers(const vecbasevector& reads, std::vector<kmer_count<(2 * K + 63) / 64>>& R, int device = 0) {
  constexpr int W = (2 * K + 63) / 64;
  Engine e(K, /*want_counts=*/true, device);
  e.AddReads(reads);
  e.Finish();
  uint64_t ni = 0, nd = 0;
  e.ck(apgk_totals(e.ctx(), &ni, &nd));
  std::vector<uint64_t> k(nd * W + 1);
  std::vector<uint32_t> c(nd + 1);
  e.ck(apgk_counts_copy(e.ctx(), 0, nd, k.data(), c.data()));
  R.resize(nd);
  for (uint64_t i = 0; i < nd; i++) {
    for (int j = 0; j < W; j++) R[i].kmer[j] = k[i * W + j];
    R[i].count = c[i];
  }
}

// One record of the full SortKmers output: one per k-mer INSTANCE.  pos is 1-based in the read and
// negative when the canonical k-mer is the reverse complement of the read's window.
template <int W>
struct kmer_record {
  uint64_t kmer[W];
  uint32_t read_id;
  int32_t pos;
};

// `SortKmers`, record form: every instance, ascending by k-mer, ties by (read id, position).
template <int K>
void SortKmers(const vecbasevector& reads, std::vector<kmer_record<(2 * K + 63) / 64>>& R, int device = 0) {
  constexpr int W = (2 * K + 63) / 64;
  Engine e(K, /*want_counts=*/true, device);
  e.AddReads(reads);
  e.Finish();
  e.ck(apgk_build_occurrences(e.ctx()));
  uint64_t ni = 0, nd = 0;
  e.ck(apgk_totals(e.ctx(), &ni, &nd));
  std::vector<uint64_t> k(nd * W + 1), off(nd + 1);
  std::vector<uint32_t> id(ni + 1);
  std::vector<int32_t> pos(ni + 1);
  e.ck(apgk_counts_copy(e.ctx(), 0, nd, k.data(), nullptr));
  e.ck(apgk_occurrences_copy(e.ctx(), 0, nd, off.data(), id.data(), pos.data()));
  R.resize(ni);
  for (uint64_t i = 0; i < nd; i++)
    for (uint64_t s = off[i]; s < off[i + 1]; s++) {
      for (int j = 0; j < W; j++) R[s].kmer[j] = k[i * W + j];
      R[s].read_id = id[s];
      R[s].pos = pos[s];
    }
}

// `KmerParcelsBuilder`: construct, Build(), then read totals / spectrum / records / batches.
class KmerParcelsBuilder {
 public:
  KmerParcelsBuilder(int K, const vecbasevector& reads, int /*n_threads: the GPU decides*/ = 0, int device = 0)
      : e_(K, true, device) { e_.AddReads(reads); }
  void Build() { e_.Finish(); built_ = true; }
  uint64_t NumKmersDistinct() const { uint64_t a, b; e_.ck(apgk_totals(e_.ctx(), &a, &b)); return b; }
  uint64_t NumKmerInstances() const { uint64_t a, b; e_.ck(apgk_totals(e_.ctx(), &a, &b)); return a; }
  KmerSpectrum Spectrum() const { KmerSpectrum s(e_.K()); s.FromEngine(e_); return s; }
  // records [first, first+n): kmers_out holds n*W words
  void Records(uint64_t first, uint64_t n, uint64_t* kmers_out, uint32_t* counts_out) const {
    e_.ck(apgk_counts_copy(e_.ctx(), first, n, kmers_out, counts_out));
  }
  // batches of k-mers [first, first+n): k-mer first+i occurs at (read_ids, positions)[run_off[i]-run_off[0] ...
  // run_off[i+1]-run_off[0]); run_off has n+1 entries
  void Batches(uint64_t first, uint64_t n, std::vector<uint64_t>& run_off, std::vector<uint32_t>& read_ids,
               std::vector<int32_t>& positions) {
    if (!occ_) { e_.ck(apgk_build_occurrences(e_.ctx())); occ_ = true; }
    run_off.assign(n + 1, 0);
    e_.ck(apgk_occurrences_copy(e_.ctx(), first, n, run_off.data(), nullptr, nullptr));
    const uint64_t m = run_off[n] - run_off[0];
    read_ids.assign(m + 1, 0); positions.assign(m + 1, 0);
    e_.ck(apgk_occurrences_copy(e_.ctx(), first, n, nullptr, read_ids.data(), positions.data()));
    read_ids.resize(m); positions.resize(m);
  }
  // affixes of k-mers [first, first+n): out[i] = bases preceding (bits 0-3) and following (bits 4-7) k-mer first+i
  void Affixes(uint64_t first, uint64_t n, uint8_t* out) {
    if (!aff_) { e_.ck(apgk_build_affixes(e_.ctx(), nullptr)); aff_ = true; }
    e_.ck(apgk_affixes_copy(e_.ctx(), first, n, out));
  }
  const Engine& engine() const { return e_; }

 private:
  Engine e_;
  bool built_ = false, occ_ = false, aff_ = false;
};

// One record of naif_kmer's "k-mer + frequency + affixes" kind (KmerFreqAffixes [U]): bit b of affixes = base b
// precedes the canonical k-mer somewhere in the reads, bit 4+b = base b follows it (include/apgk.h).
template <int W>
struct kmer_freq_affixes {
  uint64_t kmer[W];
  uint32_t count;
  uint8_t affixes;
};

// `KmerFreqAffixes`: every distinct canonical k-mer, ascending, with its count and affixes.
template <int K>
void KmerFreqAffixes(const vecbasevector& reads, std::vector<kmer_freq_affixes<(2 * K + 63) / 64>>& R, int device = 0) {
  constexpr int W = (2 * K + 63) / 64;
  Engine e(K, /*want_counts=*/true, device);
  e.AddReads(reads);
  e.Finish();
  e.ck(apgk_build_affixes(e.ctx(), nullptr));
  uint64_t ni = 0, nd = 0;
  e.ck(apgk_totals(e.ctx(), &ni, &nd));
  std::vector<uint64_t> k(nd * W + 1);
  std::vector<uint32_t> c(nd + 1);
  std::vector<uint8_t> a(nd + 1);
  e.ck(apgk_counts_copy(e.ctx(), 0, nd, k.data(), c.data()));
  e.ck(apgk_affixes_copy(e.ctx(), 0, nd, a.data()));
  R.resize(nd);
  for (uint64_t i = 0; i < nd; i++) {
    for (int j = 0; j < W; j++) R[i].kmer[j] = k[i * W + j];
    R[i].count = c[i];
    R[i].affixes = a[i];
  }
}

// The k-mer frequency table error correction queries.
class KmerFreqTable {
 public:
  KmerFreqTable(int K, const vecbasevector& reads, int device = 0) : e_(K, true, device) {
    e_.AddReads(reads);
    e_.Finish();
    e_.ck(apgk_read_store_info(e_.ctx(), &total_bases_, nullptr));
  }
  // frequency of one k-mer given as W words (canonicalised inside)
  uint32_t Freq(const uint64_t* kmer_words) const {
    uint32_t c = 0;
    e_.ck(apgk_lookup(e_.ctx(), kmer_words, 1, 1, &c));
    return c;
  }
  std::vector<uint32_t> Freqs(const std::vector<uint64_t>& kmer_words) const {
    const uint64_t n = kmer_words.size() / e_.W();
    std::vector<uint32_t> c(n);
    e_.ck(apgk_lookup(e_.ctx(), kmer_words.data(), n, 1, c.data()));
    return c;
  }
  // frequency of the window starting at every base of the reads (0xFFFFFFFF past a read's end)
  std::vector<uint32_t> ReadFreqs() const {
    std::vector<uint32_t> f(total_bases_);
    e_.ck(apgk_read_freqs(e_.ctx(), 0, total_bases_, f.data()));
    return f;
  }

 private:
  Engine e_;
  uint64_t total_bases_ = 0;
};

}  // namespace apgk_ref
