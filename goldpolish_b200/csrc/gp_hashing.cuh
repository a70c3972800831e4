// k-mer hashing shared by the filter-build kernels: byte tables, per-stream constants, and the
// "32 k-mer starts from two packed words" step (ntHash: bcgsc/goldpolish lib/nthash.hpp).
#pragma once

#include "gp_common.cuh"
#include "gp_kernels.cuh"

#include <type_traits>

namespace gp {

// byte tables for hashing 4 packed bases at a time; k-independent because groups are counted
// from the k-mer end for the forward strand and from its start for the reverse strand.
//   tf[g][b] = XOR_j srol^{4g+3-j}(seed[code_j(b)])      (bases 4 apart from the end)
//   tr[m][b] = XOR_j srol^{4m+j}(seed[3-code_j(b)])      (complement strand)
__device__ __forceinline__ void fill_hash_tables(uint64_t* tf, uint64_t* tr)
{
  for (uint32_t e = threadIdx.x; e < 8u * 256u; e += blockDim.x) {
    const uint32_t g = e >> 8, b = e & 255u;
    uint64_t f = 0, r = 0;
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) {
      const uint32_t code = (b >> (2 * j)) & 3u;
      f ^= srol(seed_of_code(code), 4 * g + 3 - j);
      r ^= srol(seed_of_code(3u - code), 4 * g + j);
    }
    tf[e] = f;
    tr[e] = r;
  }
}

// Per-lane registers that hold 32 consecutive packed / mask words of the current read (one word
// per lane) and the 32 that follow; see hash_step.
struct SeqRegs {
  uint64_t pk_cur, pk_nxt;
  uint32_t nm_cur, nm_nxt;
};

struct StreamConsts {
  uint32_t k, kq, kmask;
  uint64_t mul1, mul2, mul3;
};
__device__ __forceinline__ StreamConsts stream_consts(uint32_t k)
{
  StreamConsts c;
  c.k = k; c.kq = k >> 2;
  c.kmask = k >= 32 ? 0xFFFFFFFFu : ((1u << k) - 1u);
  c.mul1 = 1ull ^ (uint64_t(k) * kMultiSeed);
  c.mul2 = 2ull ^ (uint64_t(k) * kMultiSeed);
  c.mul3 = 3ull ^ (uint64_t(k) * kMultiSeed);
  return c;
}

// Once per stream: f(std::true_type) when k is not a multiple of 4 (its last byte is partial, see hash_kmer), else
// f(std::false_type).  The k-mer loops take the shape as a template argument, so that the usual k values run the very
// lookups they ran before other k were supported, with no per-k-mer test of the shape.
template<typename F>
__device__ __forceinline__ void with_kmer_shape(const StreamConsts& sc, F&& f)
{
  if (sc.k & 3u) f(std::true_type{});
  else f(std::false_type{});
}

// PAD > 0: the k-mer is 4 * KQ - PAD bases long and the top PAD bases of its last byte are read as A (code 0)
template<int KQ, int PAD>
__device__ __forceinline__ void hash_bytes(const uint64_t* __restrict__ tf, const uint64_t* __restrict__ tr, uint64_t w,
                                           uint64_t& fh, uint64_t& rh)
{
  uint64_t f[KQ], r[KQ];
#pragma unroll
  for (int m = 0; m < KQ; m++) {
    const uint32_t b = uint32_t(w >> (8 * m)) & (m == KQ - 1 ? 255u >> (2 * PAD) : 255u);
    f[m] = tf[((KQ - 1 - m) << 8) | b];
    r[m] = tr[(m << 8) | b];
  }
  fh = 0; rh = 0;
#pragma unroll
  for (int m = 0; m < KQ; m++) { fh ^= f[m]; rh ^= r[m]; }
}

// inverse of srol(v, s), s < 31
__host__ __device__ constexpr uint64_t sror(uint64_t v, uint32_t s)
{
  return s == 0 ? v : (((((v >> 33) >> s) | ((v >> 33) << (31u - s))) & 0x7FFFFFFFULL) << 33) |
                      ((((v & 0x1FFFFFFFFULL) >> s) | ((v & 0x1FFFFFFFFULL) << (33u - s))) & 0x1FFFFFFFFULL);
}

// canonical hash of the K-mer at the low end of w.  K = 4 * KQ - PAD with PAD in 1..3 is hashed as the 4 * KQ-mer whose
// last PAD bases are A (hash_bytes<KQ, PAD> masks them to code 0), then corrected:
//   forward  the padding adds XOR_{d<PAD} srol^d(seedA) and lifts every base's rotation by PAD:
//            fwd_K = sror^PAD(fwd_ext ^ cf)
//   reverse  the padding adds XOR_{i=K}^{4KQ-1} srol^i(seedT) (the complement of A) and leaves the bases in place:
//            rev_K = rev_ext ^ cr
// Both constants follow from K, so every K gets its own fully unrolled case (hash_h0) and a multiple of 4 runs the
// plain lookups with no correction at all.
template<int K>
__device__ __forceinline__ uint64_t hash_kmer(const uint64_t* __restrict__ tf, const uint64_t* __restrict__ tr, uint64_t w)
{
  constexpr int KQ = (K + 3) / 4, PAD = 4 * KQ - K;
  uint64_t fh, rh;
  hash_bytes<KQ, PAD>(tf, tr, w, fh, rh);
  if constexpr (PAD == 0) {
    return fh + rh;
  } else {
    constexpr uint64_t cf = srol(kSeedA, 0) ^ (PAD > 1 ? srol(kSeedA, 1) : 0ULL) ^ (PAD > 2 ? srol(kSeedA, 2) : 0ULL);
    constexpr uint64_t cr = srol(kSeedT, K) ^ (PAD > 1 ? srol(kSeedT, K + 1) : 0ULL) ^ (PAD > 2 ? srol(kSeedT, K + 2) : 0ULL);
    return sror(fh ^ cf, PAD) + (rh ^ cr);
  }
}

// Hash the k-mer that starts at position p0 + lane of the current read: validity from the mask
// window, 4 bases per table lookup (all 16 lookups independent), the 3 derived hashes, then the
// counter indices (mod 10485760) and filter bit indices (mod 2^22).
template<bool PARTIAL>
__device__ __forceinline__ bool hash_from_words(const uint64_t* __restrict__ tf, const uint64_t* __restrict__ tr,
                                                uint64_t w0, uint64_t w1, uint32_t m0, uint32_t m1, uint32_t p0,
                                                uint32_t npos, uint32_t lane, const StreamConsts& sc, uint32_t (&ci)[4],
                                                uint32_t (&bi)[4], uint64_t* h0_out = nullptr);

template<bool PARTIAL>
__device__ __forceinline__ bool hash_step(const uint64_t* __restrict__ tf, const uint64_t* __restrict__ tr,
                                          const SeqRegs& sr, uint32_t step, uint32_t p0, uint32_t npos, uint32_t lane,
                                          const StreamConsts& sc, uint32_t (&ci)[4], uint32_t (&bi)[4])
{
  const uint32_t sidx = step & 31u;
  const uint64_t w0 = __shfl_sync(0xffffffffu, sr.pk_cur, sidx);
  const uint32_t m0 = __shfl_sync(0xffffffffu, sr.nm_cur, sidx);
  uint64_t w1;
  uint32_t m1;
  if (sidx == 31u) { w1 = __shfl_sync(0xffffffffu, sr.pk_nxt, 0); m1 = __shfl_sync(0xffffffffu, sr.nm_nxt, 0); }
  else { w1 = __shfl_sync(0xffffffffu, sr.pk_cur, sidx + 1); m1 = __shfl_sync(0xffffffffu, sr.nm_cur, sidx + 1); }
  return hash_from_words<PARTIAL>(tf, tr, w0, w1, m0, m1, p0, npos, lane, sc, ci, bi);
}

// the canonical hash h0 of the k-mer starting at position p0 + lane, from packed words w0|w1 and mask words
// m0|m1 that hold positions p0 .. p0+63; false (h0 untouched) when the k-mer holds a non-ACGT base or starts
// beyond the last k-mer of the read.  PARTIAL: k is not a multiple of 4 (with_kmer_shape)
template<bool PARTIAL>
__device__ __forceinline__ bool hash_h0(const uint64_t* __restrict__ tf, const uint64_t* __restrict__ tr, uint64_t w0,
                                        uint64_t w1, uint32_t m0, uint32_t m1, uint32_t p0, uint32_t npos, uint32_t lane,
                                        const StreamConsts& sc, uint64_t& h0)
{
  const uint32_t mw = __funnelshift_r(m0, m1, lane);
  const bool valid = (p0 + lane < npos) && ((mw & sc.kmask) == 0u);
  const uint64_t w = lane ? ((w0 >> (2 * lane)) | (w1 << (64 - 2 * lane))) : w0;
  if (valid) {
    // k is uniform per stream: pick the fully unrolled lookup of this k (no per-byte branches)
    if constexpr (!PARTIAL) {
      switch (sc.kq) {
      case 8: h0 = hash_kmer<32>(tf, tr, w); break;
      case 7: h0 = hash_kmer<28>(tf, tr, w); break;
      case 6: h0 = hash_kmer<24>(tf, tr, w); break;
      case 5: h0 = hash_kmer<20>(tf, tr, w); break;
      case 4: h0 = hash_kmer<16>(tf, tr, w); break;
      case 3: h0 = hash_kmer<12>(tf, tr, w); break;
      case 2: h0 = hash_kmer<8>(tf, tr, w); break;
      default: h0 = hash_kmer<4>(tf, tr, w); break;
      }
    } else {
      switch (sc.k) {
#define GP_HASH_CASE(K) case K: h0 = hash_kmer<K>(tf, tr, w); break;
        GP_HASH_CASE(31) GP_HASH_CASE(30) GP_HASH_CASE(29) GP_HASH_CASE(27) GP_HASH_CASE(26) GP_HASH_CASE(25)
        GP_HASH_CASE(23) GP_HASH_CASE(22) GP_HASH_CASE(21) GP_HASH_CASE(19) GP_HASH_CASE(18) GP_HASH_CASE(17)
        GP_HASH_CASE(15) GP_HASH_CASE(14) GP_HASH_CASE(13) GP_HASH_CASE(11) GP_HASH_CASE(10) GP_HASH_CASE(9)
        GP_HASH_CASE(7) GP_HASH_CASE(6)
#undef GP_HASH_CASE
      default: h0 = hash_kmer<5>(tf, tr, w); break;
      }
    }
  }
  return valid;
}

// ... and its 3 derived hashes, counter indices (mod 10485760) and filter bit indices (mod 2^22)
template<bool PARTIAL>
__device__ __forceinline__ bool hash_from_words(const uint64_t* __restrict__ tf, const uint64_t* __restrict__ tr,
                                                uint64_t w0, uint64_t w1, uint32_t m0, uint32_t m1, uint32_t p0,
                                                uint32_t npos, uint32_t lane, const StreamConsts& sc, uint32_t (&ci)[4],
                                                uint32_t (&bi)[4], uint64_t* h0_out)
{
  uint64_t h0 = 0;
  const bool valid = hash_h0<PARTIAL>(tf, tr, w0, w1, m0, m1, p0, npos, lane, sc, h0);
  ci[0] = 0xFFFFFFF0u; ci[1] = 0xFFFFFFF1u; ci[2] = 0xFFFFFFF2u; ci[3] = 0xFFFFFFF3u;
  bi[0] = bi[1] = bi[2] = bi[3] = 0u;
  if (valid) {
    if (h0_out) *h0_out = h0;
    uint64_t h1 = h0 * sc.mul1, h2 = h0 * sc.mul2, h3 = h0 * sc.mul3;
    h1 ^= h1 >> kMultiShift; h2 ^= h2 >> kMultiShift; h3 ^= h3 >> kMultiShift;
    ci[0] = cbf_index(h0); ci[1] = cbf_index(h1); ci[2] = cbf_index(h2); ci[3] = cbf_index(h3);
    bi[0] = bf_index(h0); bi[1] = bf_index(h1); bi[2] = bf_index(h2); bi[3] = bf_index(h3);
  }
  return valid;
}

} // namespace gp
