// C++ host test of the affix records of include/apgk_adapters.hpp (KmerFreqAffixes, KmerParcelsBuilder::Affixes).
// Checks the hand vectors of the affix definition (include/apgk.h), then builds the records of a small random read
// set both ways and requires the same k-mers, counts and affixes, with every affix bit backed by a (K+1)-mer that
// occurs in the reads.  Prints "AFFIXES OK" and exits 0 on success.
#include <cstdio>
#include <cstdlib>
#include <random>
#include <set>
#include <string>
#include "apgk_adapters.hpp"

#define REQUIRE(c) do { if (!(c)) { std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

static std::string revcomp(const std::string& s) {
  std::string r(s.rbegin(), s.rend());
  for (char& ch : r) ch = ch == 'A' ? 'T' : ch == 'C' ? 'G' : ch == 'G' ? 'C' : 'A';
  return r;
}

int main() {
  using namespace apgk_ref;
  {  // ACGT, K=2: AC followed by G (0x40); the palindrome CG preceded by A and followed by T (0x81)
    vecbasevector r; r.push_back("ACGT");
    std::vector<kmer_freq_affixes<1>> R;
    KmerFreqAffixes<2>(r, R);
    REQUIRE(R.size() == 2);
    REQUIRE(R[0].kmer[0] == 1 && R[0].count == 2 && R[0].affixes == 0x40);
    REQUIRE(R[1].kmer[0] == 6 && R[1].count == 1 && R[1].affixes == 0x81);
  }
  for (const char* s : {"AACC", "GGTT"}) {  // K=3, a read and its reverse complement: AAC = 0x20, ACC = 0x01
    vecbasevector r; r.push_back(s);
    std::vector<kmer_freq_affixes<1>> R;
    KmerFreqAffixes<3>(r, R);
    REQUIRE(R.size() == 2);
    REQUIRE(R[0].kmer[0] == 1 && R[0].affixes == 0x20);
    REQUIRE(R[1].kmer[0] == 5 && R[1].affixes == 0x01);
  }
  {  // a read of exactly K bases has no neighbours
    vecbasevector r; r.push_back("GATTACA");
    std::vector<kmer_freq_affixes<1>> R;
    KmerFreqAffixes<7>(r, R);
    REQUIRE(R.size() == 1 && R[0].count == 1 && R[0].affixes == 0);
  }
  {  // random reads, K = 21: the adapter record form against the parcels builder, and every bit against the (K+1)-mers
    constexpr int K = 21;
    std::mt19937_64 rng(7);
    std::vector<std::string> reads;
    vecbasevector r;
    for (int i = 0; i < 300; i++) {
      std::string s;
      const int len = (int)(rng() % 60);
      for (int j = 0; j < len; j++) s += "ACGT"[rng() & 3];
      reads.push_back(s);
      r.push_back(s);
    }
    std::set<std::string> kp1;   // every (K+1)-mer of the reads, both strands
    for (const std::string& s : reads)
      for (size_t p = 0; p + K + 1 <= s.size(); p++) { kp1.insert(s.substr(p, K + 1)); kp1.insert(revcomp(s.substr(p, K + 1))); }
    std::vector<kmer_freq_affixes<1>> R;
    KmerFreqAffixes<K>(r, R);
    KmerParcelsBuilder b(K, r);
    b.Build();
    REQUIRE(b.NumKmersDistinct() == R.size() && !R.empty());
    std::vector<uint64_t> k(R.size());
    std::vector<uint32_t> c(R.size());
    std::vector<uint8_t> a(R.size());
    b.Records(0, R.size(), k.data(), c.data());
    b.Affixes(0, R.size(), a.data());
    uint64_t bits = 0;
    for (size_t i = 0; i < R.size(); i++) {
      REQUIRE(R[i].kmer[0] == k[i] && R[i].count == c[i] && R[i].affixes == a[i]);
      std::string km;
      for (int j = K - 1; j >= 0; j--) km += "ACGT"[(k[i] >> (2 * j)) & 3];
      for (int base = 0; base < 4; base++) {
        const std::string ch(1, "ACGT"[base]);
        REQUIRE(((a[i] >> base) & 1) == (kp1.count(ch + km) ? 1 : 0));
        REQUIRE(((a[i] >> (4 + base)) & 1) == (kp1.count(km + ch) ? 1 : 0));
      }
      bits += __builtin_popcount(a[i]);
    }
    REQUIRE(bits > 0);
  }
  std::printf("AFFIXES OK\n");
  return 0;
}
