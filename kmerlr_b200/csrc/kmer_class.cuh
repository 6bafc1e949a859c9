// kmer_class.cuh -- the class of one k-mer instance, as the sort-based extraction (gapped.cu) counts it and the
// generalised window scorer (score.cu) scores it.  Both include this header, so the two cannot drift apart.
//   * gapped nucleotide alphabet {a, c, g, t, n}: every instance contributes all its variants in which a subset of
//     the INTERIOR positions 1 .. k-2 is replaced by the wildcard n (those with at most max_ambiguous wildcards);
//     codes are base-5 numbers, and n is its own complement;
//   * nucleotide alphabet: one variant, base-4 codes;
//   * class = min over the variant and every enabled image (complement, reverse, revcomp; any subset of them).
// Codes fit 32 bits: 4^14 < 2^32 and 5^11 < 2^32.
#pragma once

#include <cstdint>

namespace kl {

constexpr uint32_t KMER_NONE = 0xFFFFFFFFu;   // a variant that does not count (too many wildcards)

struct ClassRule {
  int A;                             // alphabet size: 5 = gapped (wildcard variants), 4 = nucleotide
  int max_amb;                       // gapped: most wildcards per variant, -1 = no limit
  int complement, reverse, revcomp;
};

// number of wildcard masks of a k-mer (variants before the max_ambiguous filter)
__host__ __device__ __forceinline__ uint32_t kmer_masks(const ClassRule &R, int k) {
  return (R.A == 5 && k >= 2) ? 1u << (k - 2) : 1u;
}

__device__ __forceinline__ uint32_t kmer_comp(uint32_t d) { return d < 4u ? 3u - d : d; }

// class code of variant `mask` of the k-mer whose letters are the 2-bit fields of e (letter j in bits 2j, 2j+1)
__device__ __forceinline__ uint32_t kmer_variant_class(const ClassRule &R, uint32_t e, int k, uint32_t mask) {
  if (R.max_amb >= 0 && __popc(mask) > R.max_amb) return KMER_NONE;
  const int nin = (R.A == 5 && k >= 2) ? k - 2 : 0;
  auto digit = [&](int j) -> uint32_t {
    return (j >= 1 && j <= nin && ((mask >> (j - 1)) & 1u)) ? 4u : (e >> (2 * j)) & 3u;
  };
  const uint32_t A = (uint32_t)R.A;
  uint32_t c0 = 0, cc = 0, cr = 0, crc = 0;
  for (int j = 0; j < k; j++) {
    const uint32_t d = digit(j), r = digit(k - 1 - j);
    c0 = c0 * A + d;
    cc = cc * A + kmer_comp(d);                 // complement keeps the order
    cr = cr * A + r;                            // reverse keeps the letters
    crc = crc * A + kmer_comp(r);
  }
  if (R.complement && cc < c0) c0 = cc;
  if (R.reverse && cr < c0) c0 = cr;
  if (R.revcomp && crc < c0) c0 = crc;
  return c0;
}

}  // namespace kl
