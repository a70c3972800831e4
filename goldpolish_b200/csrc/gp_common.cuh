// Shared device/host definitions for the goldpolish_b200 kernels (sm_100a).
//
// ntHash arithmetic: bcgsc/goldpolish subprojects/ntedit/lib/nthash.hpp (seeds :21-28, split
// 31/33 rotation :76-97, canonical = fwd + rev :180-191, extra hashes :297-301).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace gp {

constexpr uint64_t kSeedA = 0x3c8bfbb395c60474ULL;
constexpr uint64_t kSeedC = 0x3193c18562a02b4cULL;
constexpr uint64_t kSeedG = 0x20323ed082572324ULL;
constexpr uint64_t kSeedT = 0x295549f54be24456ULL;
constexpr uint64_t kMultiSeed = 0x90b45d39fb6da1faULL;
constexpr int kMultiShift = 27;

constexpr uint64_t kCbfCounters = 10485760ULL; // 5 * 2^21
constexpr uint64_t kBfBytes = 524288ULL;
constexpr uint64_t kBfBits = kBfBytes * 8ULL;  // 2^22
constexpr uint32_t kBfWords = uint32_t(kBfBytes / 4);
constexpr int kHashNum = 4;
constexpr int kMaxK = 8;

// 2-bit codes of the packed read store
__host__ __device__ __forceinline__ uint64_t seed_of_code(uint32_t c)
{
  return c == 0 ? kSeedA : c == 1 ? kSeedC : c == 2 ? kSeedG : kSeedT;
}

// seedTab[c] on a raw byte (nthash.hpp:30-63)
__host__ __device__ __forceinline__ uint64_t seed_of_char(uint32_t c)
{
  switch (c) {
  case 1: return kSeedT;
  case 3: return kSeedG;
  case 4: return kSeedA;
  case 7: return kSeedC;
  case 'A': case 'a': return kSeedA;
  case 'C': case 'c': return kSeedC;
  case 'G': case 'g': return kSeedG;
  case 'T': case 't': return kSeedT;
  default: return 0;
  }
}
// seedTab[c & cpOff] (nthash.hpp:116): complement slot, taken from the low 3 bits of the raw byte
__host__ __device__ __forceinline__ uint64_t cseed_of_char(uint32_t c)
{
  switch (c & 7u) {
  case 1: return kSeedT;
  case 3: return kSeedG;
  case 4: return kSeedA;
  case 7: return kSeedC;
  default: return 0;
  }
}

// rotate the high 31 and the low 33 bits left by one, independently (rol1 + swapbits033)
__host__ __device__ __forceinline__ uint64_t srol1(uint64_t v)
{
  const uint64_t m = ((v & 0x8000000000000000ULL) >> 30) | ((v & 0x100000000ULL) >> 32);
  return ((v << 1) & 0xFFFFFFFDFFFFFFFFULL) | m;
}
// inverse (ror1 + swapbits3263)
__host__ __device__ __forceinline__ uint64_t sror1(uint64_t v)
{
  const uint64_t m = ((v & 0x200000000ULL) << 30) | ((v & 1ULL) << 32);
  return ((v >> 1) & 0x7FFFFFFEFFFFFFFFULL) | m;
}
// rotate both halves left by s
__host__ __device__ __forceinline__ constexpr uint64_t srol(uint64_t v, uint32_t s)
{
  const uint32_t a = s % 31u, b = s % 33u;
  uint64_t hi = v >> 33, lo = v & 0x1FFFFFFFFULL;
  hi = ((hi << a) | (hi >> (31u - a))) & 0x7FFFFFFFULL;
  lo = ((lo << b) | (lo >> (33u - b))) & 0x1FFFFFFFFULL;
  return (hi << 33) | lo;
}

struct HashState {
  uint64_t fh, rh;
};

// rolling update on raw bytes (nthash.hpp:122-131, 143-152); srol_k_* are srol(seed, k) of the
// outgoing / incoming byte, computed by the caller so that k stays a runtime value
__host__ __device__ __forceinline__ void hs_roll(HashState& h, uint32_t k, uint32_t out, uint32_t in)
{
  h.fh = srol1(h.fh) ^ seed_of_char(in) ^ srol(seed_of_char(out), k);
  h.rh = sror1(h.rh ^ srol(cseed_of_char(in), k) ^ cseed_of_char(out));
}
// replace the last base (nthash.hpp:134-140, 154-169)
__host__ __device__ __forceinline__ void hs_changelast(HashState& h, uint32_t k, uint32_t out, uint32_t in)
{
  h.fh ^= seed_of_char(out) ^ seed_of_char(in);
  h.rh = sror1(srol1(h.rh) ^ srol(cseed_of_char(out), k) ^ srol(cseed_of_char(in), k));
}

// extra hashes (nthash.hpp:297-301): h_i = b * (i ^ k * multiSeed); h_i ^= h_i >> 27
__host__ __device__ __forceinline__ uint64_t extra_hash(uint64_t base, uint32_t k, uint32_t i)
{
  uint64_t t = base * (uint64_t(i) ^ (uint64_t(k) * kMultiSeed));
  return t ^ (t >> kMultiShift);
}

// h mod 10485760 (= 5 * 2^21): low 21 bits unchanged, (h >> 21) mod 5 above them
__host__ __device__ __forceinline__ uint32_t cbf_index(uint64_t h)
{
  // (h >> 21) mod 5 by folding 16-bit limbs: 2^16 == 1 (mod 5), so the 43-bit value and the sum
  // of its limbs (< 2^18) are congruent; one 32-bit remainder finishes it
  const uint64_t hi = h >> 21;
  const uint32_t lo32 = uint32_t(hi);
  const uint32_t m = ((lo32 & 0xFFFFu) + (lo32 >> 16) + uint32_t(hi >> 32)) % 5u;
  return uint32_t(h & 0x1FFFFFu) | (m << 21);
}
__host__ __device__ __forceinline__ uint32_t bf_index(uint64_t h) { return uint32_t(h) & uint32_t(kBfBits - 1); }

} // namespace gp
