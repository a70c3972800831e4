// Counting-Bloom-gated filter build, level-synchronous form (sm_100a).
//
// Same result as fill_bfs (bcgsc/goldpolish src/utils.cpp:96-123) in the reference's order,
// computed WITHOUT walking the stream in order.  The reference's update is
//     c = min over the k-mer's 4 counters;  if (c < thr) every counter equal to c becomes c+1;
//     the k-mer enters the Bloom filter iff the count after the update is >= thr.
// Give every k-mer occurrence of a stream its position t in the reference's order and let
// T_L(x) be the time at which counter x goes from L-1 to L.  Then
//     T_{L+1}(x) = min { t : occurrence t touches x,  thr(t) > L,  t > max_j T_L(x_j(t)) }
// (all four counters had reached L before t, so the minimum is >= L; those still at L move, and
// the first such occurrence is the one that moves x), and occurrence t enters the filter iff
//     t > max_j T_{thr(t)-1}(x_j(t)).
// An occurrence that fails the test at level L fails it at every higher level.  So a stream is
// Lmax = max thr rounds of: "survivors test against T_L" then "survivors atomicMin their time
// into T_{L+1}" -- order-free inside a round, which lets ALL SMs work on ONE stream, whose
// timestamp arrays (10 485 760 x 4 B each) then live in L2 instead of HBM.  Entries carry an epoch
// tag (newer epochs compare smaller, so atomicMin overwrites stale entries, and readers treat a
// stale tag as "never"), so nothing is cleared between levels or streams.
//
// Rounds and arrays.  Round 0 hashes every occurrence, races for T_1 and puts the occurrence on its
// warp's survivor list (12 bytes: the canonical hash h0 -- the other three hashes and all eight
// indices are re-derived from it -- and time | thr << 26).  List round L reads T_L, and the
// survivors race for T_{L+1} right away in ANOTHER array.  T_1 has an array of its own (C); the
// levels above alternate between two more (A/B, parity chosen per stream).  That makes two
// consecutive streams independent enough to overlap: while stream s runs its LATE list rounds
// (L >= 2: a few survivors per thread, i.e. one list -> timestamp -> red latency chain per round),
// stream s+1 runs round 0 -- cut into as many parts as s has late rounds left -- and then its
// level-1 round beside the LAST round of s (which only reads).  One grid barrier per interval
// serves both streams; half of the warps of a CTA start with the late round, the other half with
// the head work, so that the latency chain of one hides under the instruction stream of the other.
// Every CTA takes the same deterministic sequence of decisions from uniform data.
#include "gp_hashing.cuh"

#include <algorithm>
#include <cstdlib>

namespace gp {

// list entries: time in the low 26 bits of the meta word, thr above
constexpr uint32_t kTimeBits = 26;
constexpr uint32_t kTimeMask = (1u << kTimeBits) - 1u;
// timestamp entries: tag << time_bits | time, where time_bits (LevelParams) is just wide enough for the longest
// stream of the launch: 26 bits leave 62 epochs between two clear rounds, 22 bits (3 M k-mers) a thousand.
// Tags count down (newer epochs compare smaller); the all-ones tag (epoch 0) is the cleared state.
constexpr int kLevelWarps = 8;

// A step is 32 consecutive k-mer starts of one read; steps of a stream are numbered in the
// reference's order, which makes (step * 32 + lane) the occurrence time.  A warp's share of a stream is a
// fraction [cum[0], cum[1]) of it -- equal fractions to begin with, then proportional to the speed measured for
// the warp's SM (the same work takes 88..106 us depending on where the SM sits) -- cut into kRuns runs that are
// spread over the whole time axis: the stream is kRuns "rows" (time slabs) and the warp takes its fraction of
// every row, the row boundaries dithered by r / kRuns so that the roundings of the rows do not add up (at
// 5 steps per warp every row gives a warp 0 or 1 step).  Survivors crowd towards late times; contiguous shares
// left the early warps idle in every list round.  anchor[] maps a step to its read entry; lane r fetches the
// head of run r, so that the dependent loads of all runs overlap.
constexpr uint32_t kRuns = 8;

struct LevelCtx {
  const uint64_t* tf;
  const uint64_t* tr;
  uint32_t lane, gwarp;
};

// steps before the warp's share (its survivor list starts there, + one slack slot per row and warp)
__device__ __forceinline__ uint64_t warp_list_base(uint32_t n_steps, const uint64_t* cum, uint32_t gwarp)
{
  return ((uint64_t(n_steps) * cum[0]) >> 32) + uint64_t(gwarp) * (kRuns + 1u);
}
// run of row r (0..kRuns-1) of this warp: first step and length (0: none)
__device__ __forceinline__ void run_of_row(uint32_t r, uint32_t n_steps, const uint64_t* cum, uint32_t& s0, uint32_t& len)
{
  const uint32_t r0 = uint32_t(uint64_t(n_steps) * r / kRuns), r1 = uint32_t(uint64_t(n_steps) * (r + 1u) / kRuns);
  const uint64_t rowlen = r1 - r0, phase = (uint64_t(r) << 32) / kRuns;
  // boundaries floor(rowlen * cum + phase): 0 for cum = 0, rowlen for cum = 2^32, the same on both sides of a warp border
  const uint32_t a = uint32_t((rowlen * cum[0] + phase) >> 32), b = uint32_t((rowlen * cum[1] + phase) >> 32);
  s0 = r0 + a;
  len = r < kRuns ? b - a : 0u;
}

// h0 -> the four hashes' counter indices (mod 10485760), each with bit 21 of its hash on top (bit 24), so that
// the 22-bit filter index is recoverable from the same word
__device__ __forceinline__ uint32_t pack_index(uint64_t h) { return cbf_index(h) | ((uint32_t(h >> 21) & 1u) << 24); }
__device__ __forceinline__ void unpack_index(uint32_t w, uint32_t& ci, uint32_t& bi)
{
  ci = w & 0xFFFFFFu;
  bi = (w & 0x1FFFFFu) | ((w >> 24) << 21);
}
__device__ __forceinline__ void derive_rest(uint64_t h0, const StreamConsts& sc, uint32_t (&pw)[4])
{ // nthash.hpp:297-301
  uint64_t h1 = h0 * sc.mul1, h2 = h0 * sc.mul2, h3 = h0 * sc.mul3;
  h1 ^= h1 >> kMultiShift; h2 ^= h2 >> kMultiShift; h3 ^= h3 >> kMultiShift;
  pw[1] = pack_index(h1); pw[2] = pack_index(h2); pw[3] = pack_index(h3);
}

// Calls f(step, entry thr, valid, h0, pw) for every step of this warp's runs in rows [row0, row1).
template<bool PARTIAL, typename F>
__device__ __forceinline__ void for_runs(const LevelParams& p, const LevelCtx& c, const uint64_t* cum, uint32_t batch, uint32_t ki,
                                         const StreamConsts& sc, uint32_t n_steps, uint32_t row0, uint32_t row1, F&& f)
{
  const uint32_t* pre = p.step_pre + uint64_t(ki) * (p.n_entries + 1);
  const uint64_t e0 = p.batch_entry_off[batch], e1 = p.batch_entry_off[batch + 1];
  const uint32_t base = __ldg(pre + e0);
  const uint16_t* anchor = p.anchor + uint64_t(ki) * p.anchor_stride + base;
  uint32_t h_e = 0, h_first = 0, h_last = 0, h_thr = 0, h_len = 0, h_wlo = 0, h_whi = 0;
  {
    uint32_t s0 = 0, len = 0;
    if (c.lane >= row0 && c.lane < row1) run_of_row(c.lane, n_steps, cum, s0, len);
    if (len) {
      h_e = __ldg(anchor + s0);
      const uint64_t e = e0 + h_e;
      h_first = __ldg(pre + e) - base; h_last = __ldg(pre + e + 1) - base;
      const gp_read_entry ent = p.entries[e];
      h_thr = ent.kmer_threshold;
      h_len = p.read_len[ent.read_id];
      const uint64_t wb = p.read_boff[ent.read_id] >> 5;
      h_wlo = uint32_t(wb); h_whi = uint32_t(wb >> 32);
    }
  }
#pragma unroll 1
  for (uint32_t r = row0; r < row1; r++) {
    uint32_t s0, len;
    run_of_row(r, n_steps, cum, s0, len);
    if (len == 0) continue;
    const uint32_t s_end = s0 + len;
    const uint64_t e_head = e0 + __shfl_sync(0xffffffffu, h_e, r);
    uint32_t first = __shfl_sync(0xffffffffu, h_first, r), last = __shfl_sync(0xffffffffu, h_last, r);
    uint32_t kthr = __shfl_sync(0xffffffffu, h_thr, r), len_r = __shfl_sync(0xffffffffu, h_len, r);
    uint64_t wbase = uint64_t(__shfl_sync(0xffffffffu, h_wlo, r)) | (uint64_t(__shfl_sync(0xffffffffu, h_whi, r)) << 32);
    uint32_t s = s0;
    for (uint64_t e = e_head; e < e1 && s < s_end; e++) {
      if (e != e_head) { // the run crosses into the next read
        first = __ldg(pre + e) - base; last = __ldg(pre + e + 1) - base;
        if (last <= s) continue;
        const gp_read_entry ent = p.entries[e];
        kthr = ent.kmer_threshold;
        len_r = p.read_len[ent.read_id];
        wbase = p.read_boff[ent.read_id] >> 5;
      }
      const uint32_t thr = kthr - 2u + ki; // utils.cpp:108,121
      const uint32_t npos = len_r - sc.k + 1;
      // the words of step s+1 are requested before step s is processed
      uint32_t rs = s - first;
      uint64_t w0 = __ldg(p.pk + wbase + rs), w1 = __ldg(p.pk + wbase + rs + 1);
      uint32_t m0 = __ldg(p.nm + wbase + rs), m1 = __ldg(p.nm + wbase + rs + 1);
      for (; s < last && s < s_end; s++) {
        rs = s - first; // step within the read
        const uint64_t cw0 = w0, cw1 = w1;
        const uint32_t cm0 = m0, cm1 = m1;
        if (s + 1 < last && s + 1 < s_end) {
          w0 = cw1; m0 = cm1; // consecutive steps share a word
          w1 = __ldg(p.pk + wbase + rs + 2);
          m1 = __ldg(p.nm + wbase + rs + 2);
        }
        uint64_t h0 = 0;
        const bool valid = hash_h0<PARTIAL>(c.tf, c.tr, cw0, cw1, cm0, cm1, rs * 32u, npos, c.lane, sc, h0);
        uint32_t pw[4] = { 0xFFFFF0u, 0xFFFFF1u, 0xFFFFF2u, 0xFFFFF3u };
        if (valid) { pw[0] = pack_index(h0); derive_rest(h0, sc, pw); }
        f(s, thr, valid, h0, pw);
      }
    }
  }
}

// anchor[ki][s] = entry (relative to its batch's first entry) that holds global step s of k index ki
__global__ void fill_anchor_kernel(const uint32_t* __restrict__ step_pre, const uint16_t* __restrict__ entry_rel,
                                   uint16_t* __restrict__ anchor, uint32_t n_entries, uint32_t nk, uint64_t anchor_stride)
{
  const uint64_t w = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  if (w >= uint64_t(n_entries) * nk) return;
  const uint32_t ki = uint32_t(w / n_entries), e = uint32_t(w - uint64_t(ki) * n_entries);
  const uint32_t* pre = step_pre + uint64_t(ki) * (n_entries + 1);
  const uint32_t a = pre[e], b = pre[e + 1];
  const uint16_t v = entry_rel[e];
  for (uint32_t s = a + lane; s < b; s += 32) anchor[uint64_t(ki) * anchor_stride + s] = v;
}

void launch_fill_anchor(const uint32_t* step_pre, const uint16_t* entry_rel, uint16_t* anchor, uint32_t n_entries,
                        uint32_t nk, uint64_t anchor_stride, cudaStream_t s)
{
  const uint64_t warps = uint64_t(n_entries) * nk;
  if (warps == 0) return;
  fill_anchor_kernel<<<uint32_t((warps + 7) / 8), 256, 0, s>>>(step_pre, entry_rel, anchor, n_entries, nk, anchor_stride);
}

// Survivor lists: occurrences that passed level L.  An entry is kSurvWords = 3 words: the canonical hash h0
// (the three other hashes are multiply-xorshifts of it, nthash.hpp:297-301: ~40 instructions against 8 bytes
// of list traffic per visit) and time | thr << 26.  Lists are WARP-PRIVATE: a warp keeps the survivors of its own
// share of the stream in its own region (share * 32 entries) and compacts them in place level after level -- no
// list counters, no reservation atomics.  Two list buffers alternate between consecutive streams (the late
// rounds of one stream run beside round 0 of the next).
struct SurvList {
  uint32_t *lo, *hi, *meta;   // h0 low, h0 high, time | thr << 26; already offset to the warp's region
};
__device__ __forceinline__ SurvList list_of(const LevelParams& p, uint32_t buf, uint32_t n_steps, const uint64_t* cum, uint32_t gwarp)
{
  SurvList l;
  l.lo = p.surv + uint64_t(buf) * kLevelSurvWords * p.surv_cap + warp_list_base(n_steps, cum, gwarp) * 32u;
  l.hi = l.lo + p.surv_cap;
  l.meta = l.hi + p.surv_cap;
  return l;
}
// append the lanes with q set at position cnt of the warp's list
__device__ __forceinline__ void surv_append(const SurvList& l, uint32_t& cnt, bool q, uint64_t h0, uint32_t meta, uint32_t lane)
{
  const uint32_t m = __ballot_sync(0xffffffffu, q);
  if (q) {
    const uint32_t i = cnt + __popc(m & ((1u << lane) - 1u));
    l.lo[i] = uint32_t(h0);
    l.hi[i] = uint32_t(h0 >> 32);
    l.meta[i] = meta;
  }
  cnt += __popc(m);
}
// entries r + 32 e + lane (e < E) of a list of cnt entries; zeros beyond its end
template<int E>
__device__ __forceinline__ void fetch_entries(const SurvList& l, uint32_t cnt, uint32_t r, uint32_t lane, uint32_t (&lo)[E],
                                              uint32_t (&hi)[E], uint32_t (&meta)[E])
{
#pragma unroll
  for (int e = 0; e < E; e++) {
    const uint32_t i = r + 32u * e + lane;
    lo[e] = 0; hi[e] = 0; meta[e] = 0;
    if (i < cnt) {
      lo[e] = __ldcg(l.lo + i);
      hi[e] = __ldcg(l.hi + i);
      meta[e] = __ldcg(l.meta + i);
    }
  }
}
// fire-and-forget atomics (REDG): spelled in PTX because ptxas keeps the returning form (ATOMG
// with a dead destination) for atomicMin/atomicOr in this kernel
__device__ __forceinline__ void red_min(uint32_t* p, uint32_t v)
{
  asm volatile("red.relaxed.gpu.global.min.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_or(uint32_t* p, uint32_t v)
{
  asm volatile("red.relaxed.gpu.global.or.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ void bf_load(const uint32_t* __restrict__ bf, const uint32_t (&pw)[4], uint32_t (&w)[4])
{ // the filter is 512 KiB and mostly hit by repeats of the same k-mers: look first
#pragma unroll
  for (int j = 0; j < 4; j++) { uint32_t ci, bi; unpack_index(pw[j], ci, bi); w[j] = __ldcg(bf + (bi >> 5)); }
}
__device__ __forceinline__ void bf_set(uint32_t* __restrict__ bf, const uint32_t (&pw)[4], const uint32_t (&w)[4])
{
#pragma unroll
  for (int j = 0; j < 4; j++) {
    uint32_t ci, bi;
    unpack_index(pw[j], ci, bi);
    if (!(w[j] & (1u << (bi & 31u)))) red_or(bf + (bi >> 5), 1u << (bi & 31u));
  }
}
__device__ __forceinline__ void bf_insert(uint32_t* __restrict__ bf, const uint32_t (&pw)[4])
{
  uint32_t w[4];
  bf_load(bf, pw, w);
  bf_set(bf, pw, w);
}

// ---- list rounds ----
// One list round of one warp: who sees all four counters at >= L before its own time?  Survivors with thr = L + 1
// enter the filter and, unless it is the stream's last round, race for T_{L+1} right away in the other array; the
// list is compacted in place.  Two shapes:
//   list_round_all    every entry loads its four timestamps at once (and, if it would enter the filter in this
//                     round, the four filter words with them): one memory round trip per 64 entries.  The late
//                     rounds, and any round that materialises counter bytes.
//   list_round_first  level 1: most entries fail on their first counter (they are its first toucher); the other
//                     three are only loaded for those that do not -- fewer touches, two round trips.  (Loading
//                     all four for four entries per lane was tried for short lists: 19 against 13 us; software
//                     pipelining the two round trips over the iterations: 11.7 against 11.0 us -- the round is
//                     within 70 % of what its loads and atomics cost at the measured L2 rates.)
struct ListJob {
  SurvList lst;
  uint32_t cnt;
  const uint32_t* V;   // T_L
  uint32_t* Vn;        // where T_{L+1} goes
  uint32_t* bf;
  uint8_t* cbf;
  uint32_t L, lread, tag, tag_next, vmask;
};

__device__ __forceinline__ uint32_t list_round_all(const ListJob& J, const StreamConsts& sc, uint32_t lane, uint32_t (&nlo)[2],
                                                   uint32_t (&nhi)[2], uint32_t (&nmeta)[2])
{
  uint32_t kept = 0;
  for (uint32_t r = 0; r < J.cnt; r += 64u) {
    uint64_t h0[2];
    uint32_t pw[2][4], meta[2], v[2][4], fw[2][4];
    bool live[2], q[2], ins[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      live[e] = r + 32u * e + lane < J.cnt;
      meta[e] = nmeta[e];
      h0[e] = uint64_t(nlo[e]) | (uint64_t(nhi[e]) << 32);
      ins[e] = live[e] && (meta[e] >> kTimeBits) == J.L + 1u; // enters the filter if it survives this round
      pw[e][0] = pack_index(h0[e]);
      derive_rest(h0[e], sc, pw[e]);
#pragma unroll
      for (int j = 0; j < 4; j++) v[e][j] = live[e] ? __ldcg(J.V + (pw[e][j] & 0xFFFFFFu)) : 0u;
#pragma unroll
      for (int j = 0; j < 4; j++) fw[e][j] = 0u;
      if (ins[e]) bf_load(J.bf, pw[e], fw[e]);
    }
    // the entries of the next iteration are requested now: this iteration's appends stay below r + 64
    if (r + 64u < J.cnt) fetch_entries<2>(J.lst, J.cnt, r + 64u, lane, nlo, nhi, nmeta);
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const uint32_t t = meta[e] & kTimeMask, thr = meta[e] >> kTimeBits;
      bool reached = live[e];
      uint32_t mx = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        reached &= (v[e][j] & ~J.vmask) == J.tag;
        mx = max(mx, v[e][j] & J.vmask);
        if (J.cbf && live[e] && v[e][j] == (J.tag | t)) J.cbf[pw[e][j] & 0xFFFFFFu] = (uint8_t)J.L; // moved counter j to level L
      }
      q[e] = reached && t > mx && thr > J.L;
      if (q[e] && ins[e]) bf_set(J.bf, pw[e], fw[e]);
      if (q[e] && J.L < J.lread) {
#pragma unroll
        for (int j = 0; j < 4; j++) red_min(J.Vn + (pw[e][j] & 0xFFFFFFu), J.tag_next | t);
      }
    }
    // every lane has both entries in registers before the ballots inside return; kept <= r
    surv_append(J.lst, kept, q[0], h0[0], meta[0], lane);
    surv_append(J.lst, kept, q[1], h0[1], meta[1], lane);
  }
  return kept;
}

__device__ __forceinline__ uint32_t list_round_first(const ListJob& J, const StreamConsts& sc, uint32_t lane, uint32_t (&nlo)[2],
                                                     uint32_t (&nhi)[2], uint32_t (&nmeta)[2])
{
  uint32_t kept = 0;
  for (uint32_t r = 0; r < J.cnt; r += 64u) {
    uint64_t h0[2];
    uint32_t pw[2][4], meta[2], v0[2], v[2][3];
    bool live[2], q[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      live[e] = r + 32u * e + lane < J.cnt;
      meta[e] = nmeta[e];
      h0[e] = uint64_t(nlo[e]) | (uint64_t(nhi[e]) << 32);
      pw[e][0] = pack_index(h0[e]);
      v0[e] = live[e] ? __ldcg(J.V + (pw[e][0] & 0xFFFFFFu)) : 0u;
    }
    if (r + 64u < J.cnt) fetch_entries<2>(J.lst, J.cnt, r + 64u, lane, nlo, nhi, nmeta);
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const uint32_t t = meta[e] & kTimeMask;
      q[e] = live[e] && (v0[e] & ~J.vmask) == J.tag && (v0[e] & J.vmask) < t;
      if (q[e]) derive_rest(h0[e], sc, pw[e]);
#pragma unroll
      for (int j = 0; j < 3; j++) v[e][j] = q[e] ? __ldcg(J.V + (pw[e][j + 1] & 0xFFFFFFu)) : 0u;
    }
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const uint32_t t = meta[e] & kTimeMask, thr = meta[e] >> kTimeBits;
#pragma unroll
      for (int j = 0; j < 3; j++) q[e] = q[e] && (v[e][j] & ~J.vmask) == J.tag && (v[e][j] & J.vmask) < t;
      q[e] = q[e] && thr > J.L;
      if (q[e] && thr == J.L + 1u) bf_insert(J.bf, pw[e]);
      if (q[e] && J.L < J.lread) {
#pragma unroll
        for (int j = 0; j < 4; j++) red_min(J.Vn + (pw[e][j] & 0xFFFFFFu), J.tag_next | t);
      }
    }
    surv_append(J.lst, kept, q[0], h0[0], meta[0], lane);
    surv_append(J.lst, kept, q[1], h0[1], meta[1], lane);
  }
  return kept;
}

// ---- grid barrier: one monotone counter ----
// polling uses a relaxed load (an acquire load costs an L1 invalidate -- CCTL.IVALL -- per poll);
// one fence after the loop orders the data reads of the next round behind it
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p)
{
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ unsigned long long globaltimer_ns()
{
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// A stream's filter is final (its last barrier has drained on this CTA): stream it to the caller's pinned
// host buffer if there is one -- every CTA copies its slice straight over PCIe, under the following rounds, so
// that no bulk D2H is left at the end -- and tell the edit kernel (gp_pipeline_run).
__device__ __forceinline__ void filter_final(const LevelParams& p, uint32_t batch, uint32_t ki, uint32_t slot, uint32_t gtid, uint32_t gthreads)
{
  if (p.bf_host) {
    const uint4* __restrict__ src = reinterpret_cast<const uint4*>(p.bf_pool + (uint64_t(slot) * p.nk + ki) * kBfWords);
    uint4* __restrict__ dst = reinterpret_cast<uint4*>(p.bf_host + (uint64_t(batch) * p.nk + ki) * kBfWords);
    for (uint32_t i = gtid; i < kBfWords / 4u; i += gthreads) dst[i] = __ldcg(src + i);
  }
  if (p.batch_done && gtid == 0) {
    atomicAdd(p.batch_done + batch, 1u);
    atomicAdd(p.batch_done + p.n_batches_total, 1u); // progress beacon for the edit kernel's watchdog
  }
}

// sum over the CTA, the same value in every thread (scratch: one slot per warp)
__device__ __forceinline__ unsigned long long block_sum(unsigned long long v, unsigned long long* scratch)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31u) == 0u) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long t = 0;
  for (uint32_t w = 0; w < (blockDim.x >> 5); w++) t += scratch[w];
  return t;
}

// what the head stream does in an interval
enum : uint32_t { MK_NONE = 0, MK_CLEAR = 1, MK_R0 = 2, MK_R1 = 3 };

struct StreamSt {       // one stream in flight (uniform over the grid: every CTA derives the same values)
  uint32_t valid;
  uint32_t sid, batch, ki, n_steps, lread;
  uint32_t slot;        // where its filter lives in the pool
  uint32_t buf;         // which list buffer it uses
  uint32_t cum;         // which share table it uses
  uint32_t pb;          // T_L (L >= 2) lives in array (L + pb) & 1; T_1 in array 2, or (two arrays) in (1 + pb) & 1
  uint32_t L;           // its next list round
  uint32_t tag;         // tag carried by T_L (what round L reads)
  uint32_t tag_next;    // tag given to T_{L+1} in round L
};

struct Sched {          // the planner's own state
  StreamSt cur;         // head stream: round 0 (in parts), then its level-1 round
  StreamSt tail;        // previous stream: late list rounds (L >= 2)
  uint32_t next_sid, epoch, ord;
  uint32_t need_clear, parts, part, r0_done, publish, recal; // of cur
  uint4 nx_info;        // stream_tab entry of stream next_sid, fetched one stream ahead
};

struct Plan {           // what one interval does; written by the planner thread one interval ahead
  uint32_t finished, main_kind, tail_on;
  uint32_t row0, row1, part, last_part, publish, recal; // main_kind == MK_R0
  StreamSt cur, tail;   // snapshots valid for this interval
  uint32_t done_n, done_b[2], done_ki[2], done_slot[2]; // streams whose last round ran in the interval before
};

// 3 CTAs of 8 warps per SM (80 registers); a 64-register build with 4 CTAs spills and measured 8 % slower
__global__ void __launch_bounds__(kLevelWarps * 32, 3) build_filters_levels_kernel(LevelParams p)
{
  __shared__ uint64_t tf[8 * 256];
  __shared__ uint64_t tr[8 * 256];
  __shared__ Sched sch;
  __shared__ Plan plans[2];
  __shared__ uint32_t warp_cnt[2][kLevelWarps];         // survivors in each warp's private list, per list buffer
  __shared__ uint64_t cum_sh[2][kLevelWarps + 1];       // two tables of share boundaries of this CTA's warps (fractions of 2^32)
  __shared__ unsigned long long cal_ns, cal_steps;      // round-0 work of this CTA's first warp since its last speed publication
  __shared__ unsigned long long red_sh[3][kLevelWarps];
  __shared__ unsigned long long diag[kLevelDiag];       // interval-time diagnostics of this CTA (thread 0)
  __shared__ uint32_t dense_sh; // this CTA's number among those that build
  if (p.batch_done) asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); // the edit kernel may join us now
  // Which CTA am I, of how many?  Normally blockIdx.x of gridDim.x.  gp_pipeline_run keeps a few SMs back for the edit
  // kernel (p.keep_sms < p.sms): the launch fills EVERY SM with gridDim.x / p.sms CTAs, the CTAs of the last SMs to
  // arrive leave at once, and the edit kernel launched behind us -- CTAs that need a whole SM -- lands exactly there.
  // The two kernels then share L2 but no SM; an edit warp beside build warps slowed its SM's share of EVERY barrier
  // interval, i.e. the whole grid.  Which CTAs share an SM is the hardware's business (blockIdx.x % SMs it is not:
  // tried), and %smid is not contiguous, so the SMs are numbered in order of arrival: the first CTA on an SM draws the
  // SM's rank, the others wait for it (all CTAs are resident: cooperative launch).  The CTAs that stay are numbered
  // densely, round * keep_sms + rank: the CTAs of one SM stay far apart, as in a plain launch -- neighbouring CTAs hold
  // neighbouring pieces of every time slab (the same reads), and an SM whose three CTAs were neighbours carried three
  // times the unevenness of survivors into every interval (measured: +7 %).  The dense number lives in shared memory
  // and is read where it is needed (once per interval: the warp's list region), so that it costs no
  // register across the hot loops.
  if (threadIdx.x == 0) {
    uint32_t dense = blockIdx.x;
    if (p.keep_sms < p.sms) {
      const uint32_t per_sm = gridDim.x / p.sms;
      uint32_t smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      uint32_t* arrivals = p.sm_table + 1u + 2u * (smid & 2047u);
      uint32_t* rank_p1 = arrivals + 1;
      const uint32_t slot = atomicAdd(arrivals, 1u); // (the host checks afterwards that every SM counted per_sm)
      uint32_t rank;
      if (slot == 0u) {
        rank = atomicAdd(p.sm_table, 1u);
        atomicExch(rank_p1, rank + 1u);
      } else {
        while ((rank = *reinterpret_cast<volatile uint32_t*>(rank_p1)) == 0u) { }
        rank -= 1u;
      }
      dense = rank < p.keep_sms && slot < per_sm ? slot * p.keep_sms + rank : 0xFFFFFFFFu;
    }
    dense_sh = dense;
  }
  __syncthreads();
  if (dense_sh == 0xFFFFFFFFu) return; // an SM given back: this CTA has taken part in nothing
#define nb (p.n_ctas)
#define bid dense_sh
#define gtid (dense_sh * blockDim.x + threadIdx.x)
#define gthreads (nb * blockDim.x)
  LevelCtx c;
  c.lane = threadIdx.x & 31u;
  c.gwarp = 0; // (not used by this kernel: the warp's number among those that build is gwarp_now)
  if (bid == 0 && threadIdx.x == 0) atomicMin(p.counters + 20, globaltimer_ns()); // (several waves: the first start)
  fill_hash_tables(tf, tr);
  c.tf = tf; c.tr = tr;
#define gwarp_now (dense_sh * uint32_t(kLevelWarps) + wib)
  const uint32_t nwarps = (nb * blockDim.x) >> 5;
  const uint32_t wib = threadIdx.x >> 5;
  const uint32_t tb = p.time_bits, vmask = (1u << tb) - 1u, maxtag = (1u << (32u - tb)) - 1u;
  const bool planner = threadIdx.x == 32u; // a thread that neither polls nor arrives: planning stays off the barrier's critical path
  unsigned long long ops = 0, list_seen = 0;
  if (threadIdx.x == 0) { cal_ns = 0; cal_steps = 0; }
  if (threadIdx.x < kLevelDiag) diag[threadIdx.x] = 0;
  if (threadIdx.x <= uint32_t(kLevelWarps)) // equal shares until speeds have been measured
    cum_sh[0][threadIdx.x] = cum_sh[1][threadIdx.x] = (uint64_t(bid * kLevelWarps + threadIdx.x) << 32) / nwarps;

  // ---- scheduling (planner thread only; every CTA computes the same sequence from uniform data) ----
  auto new_tag = [&]() { sch.epoch++; return (maxtag - sch.epoch) << tb; };
  auto begin_stream = [&]() {   // next stream with work becomes the head; sch.cur.valid = 0 when there is none
    StreamSt& S = sch.cur;
    const uint32_t prev_cum = S.cum;
    S.valid = 0;
    for (;;) {
      const uint32_t sid = sch.next_sid;
      if (sid >= p.n_streams) return;
      sch.next_sid = sid + 1u;
      const uint4 info = sch.nx_info;
      if (sid + 1u < p.n_streams) sch.nx_info = __ldg(p.stream_tab + sid + 1u);
      const uint32_t ki = sid % p.nk, batch = info.z;
      if (info.x == 0) { // nothing to insert: the (zeroed) filter is final
        if (p.batch_done && bid == 0) { atomicAdd(p.batch_done + batch, 1u); atomicAdd(p.batch_done + p.n_batches_total, 1u); }
        continue;
      }
      const uint32_t lmax = info.y; // largest thr of the stream (kmer_threshold - 2 + k index, utils.cpp:108,121)
      S.valid = 1; S.sid = sid; S.batch = batch; S.ki = ki; S.n_steps = info.x;
      S.slot = p.bf_slot ? __ldg(p.bf_slot + batch) : batch;
      // levels that need a read round: up to lmax-1 for the filter bits (an insert happens at
      // L = thr-1); one more when the counter bytes themselves are wanted (who reached lmax)
      S.lread = p.cbf_pool ? lmax : lmax - 1u;
      S.buf = sch.ord & 1u;
      sch.ord++;
      sch.publish = p.weighted && (sch.ord & 63u) == 4u; // after 4 streams, then every 64: publish the CTA's speed ...
      sch.recal = p.weighted && (sch.ord & 63u) == 5u;   // ... and the next stream starts with re-weighted shares,
      S.cum = sch.recal ? prev_cum ^ 1u : prev_cum;       // in the table that the stream before it does not use
      sch.part = 0; sch.r0_done = 0;
      // the tags of this stream and of the late rounds still to come of the one before it must not wrap
      const uint32_t pending = sch.tail.valid ? sch.tail.lread + 2u - sch.tail.L : 0u;
      sch.need_clear = sch.epoch + lmax + 2u + pending > maxtag - 1u;
      // three arrays: its T_2 must not land in the array that the last round of the stream before it reads;
      // two arrays (T_1 alternates with the others): its T_1 must not
      const uint32_t z = (sch.tail.lread + sch.tail.pb) & 1u;
      S.pb = sch.tail.valid ? (p.arrays == 3u ? z ^ 1u : z) : 0u;
      // three arrays: round 0 in as many parts as the tail has late rounds left before its last one
      sch.parts = 1;
      if (p.overlap && p.arrays == 3u && sch.tail.valid && !sch.need_clear) {
        const uint32_t left = sch.tail.lread + 1u - sch.tail.L; // rounds L .. lread
        sch.parts = left > 2u ? min(left - 1u, kRuns) : 1u;
      }
      return; // (the tag of its T_1 is drawn when its round 0 starts: tags must reach every array in order)
    }
  };
  // what the interval after `prev` does (prev == nullptr: the first one)
  auto make_plan = [&](const Plan* prev, Plan& P) {
    P.done_n = 0;
    auto push_done = [&](const StreamSt& S) { P.done_b[P.done_n] = S.batch; P.done_ki[P.done_n] = S.ki; P.done_slot[P.done_n] = S.slot; P.done_n++; };
    if (prev) { // ---- advance both streams past the interval `prev` ----
      if (prev->tail_on) {
        if (sch.tail.L >= sch.tail.lread) { push_done(sch.tail); sch.tail.valid = 0; }
        else { sch.tail.L++; sch.tail.tag = sch.tail.tag_next; }
      }
      switch (prev->main_kind) {
      case MK_CLEAR:
        sch.epoch = 0; sch.need_clear = 0;
        break;
      case MK_R0:
        if (++sch.part == sch.parts) {
          sch.r0_done = 1;
          if (sch.cur.lread == 0u) { push_done(sch.cur); sch.cur.valid = 0; } // (thr <= 1 everywhere: no list round)
        }
        break;
      case MK_R1: // T_2 was written under tag_next; the stream goes on as the tail (the old tail has just finished)
        if (sch.cur.lread <= 1u) push_done(sch.cur);
        else { sch.tail = sch.cur; sch.tail.L = 2; sch.tail.tag = sch.cur.tag_next; }
        sch.cur.valid = 0;
        break;
      default: break;
      }
    }
    if (!sch.cur.valid) begin_stream();
    P.tail_on = sch.tail.valid;
    P.main_kind = MK_NONE;
    if (sch.cur.valid) {
      if (sch.need_clear) {
        if (!sch.tail.valid) P.main_kind = MK_CLEAR; // (waits for the tail: both streams' arrays are cleared)
      } else if (!sch.r0_done) {
        // two arrays: round 0 may only join the tail's LAST round (which reads one array and writes none)
        if (!sch.tail.valid || (p.overlap && (p.arrays == 3u || sch.tail.L == sch.tail.lread))) {
          P.main_kind = MK_R0;
          if (sch.part == 0u) sch.cur.tag = new_tag();
          P.part = sch.part;
          P.last_part = sch.part + 1u == sch.parts;
          P.row0 = kRuns * sch.part / sch.parts;
          P.row1 = kRuns * (sch.part + 1u) / sch.parts;
          P.publish = sch.publish; P.recal = sch.recal;
        }
      } else { // level-1 round: three arrays only, beside the LAST round of the tail (it writes T_2 into the array that round does not read)
        if (!sch.tail.valid || (p.overlap && p.arrays == 3u && sch.tail.L == sch.tail.lread)) {
          P.main_kind = MK_R1;
          sch.cur.L = 1;
          sch.cur.tag_next = new_tag();
        }
      }
    }
    if (P.tail_on) sch.tail.tag_next = new_tag();
    P.cur = sch.cur; P.tail = sch.tail;
    P.finished = P.main_kind == MK_NONE && !P.tail_on;
  };
  if (planner) {
    sch.next_sid = 0; sch.epoch = 0; sch.ord = 0; // V arrives cleared (all 0xFFFFFFFF = epoch 0)
    sch.cur.valid = 0; sch.cur.cum = 0; sch.tail.valid = 0;
    sch.need_clear = 0; sch.parts = 1; sch.part = 0; sch.r0_done = 0; sch.publish = 0; sch.recal = 0;
    sch.nx_info = p.n_streams ? __ldg(p.stream_tab) : make_uint4(0u, 0u, 0u, 0u);
    make_plan(nullptr, plans[0]);
  }
  __syncthreads();

  // T_1 of a stream: the third array, or (two arrays) the one its T_2 does not use
  auto t1_array = [&](const StreamSt& S) { return p.V + (p.arrays == 3u ? 2u : ((1u + S.pb) & 1u)) * kCbfCounters; };
  unsigned long long target = 0; // barrier count that must be reached before the coming interval (thread 0)
  for (uint32_t it = 0;; it++) {
    // Between the __syncthreads that ended the previous interval's work and the one below, plans[it & 1] is stable (it
    // was written during the previous interval), thread 0 arrives at and polls the grid barrier, and everybody else
    // fetches the first entries of its first list round -- its own list, independent of the other CTAs.
    const Plan& P = plans[it & 1u];
    const uint32_t main_kind = P.main_kind, tail_on = P.tail_on;
    // this warp runs the tail's list round first if it is an even warp, the head's work first otherwise: the
    // latency chain of a late round (few entries per thread) hides under the other half's instruction stream
    const bool tail_first = tail_on && ((wib & 1u) == 0u || main_kind == MK_NONE);
    uint32_t nx_lo[2], nx_hi[2], nx_meta[2];
    uint32_t pre_for = 0; // 1: tail list prefetched, 2: head list prefetched
    if (!P.finished && (tail_first || main_kind == MK_R1)) {
      const StreamSt* S = tail_first ? &P.tail : &P.cur;
      const SurvList l = list_of(p, S->buf, S->n_steps, cum_sh[S->cum] + wib, gwarp_now);
      fetch_entries<2>(l, warp_cnt[S->buf][wib], 0, c.lane, nx_lo, nx_hi, nx_meta);
      pre_for = tail_first ? 1u : 2u;
    }
    unsigned long long t_a = 0, t_b = 0;
    if (threadIdx.x == 0) {
      t_a = globaltimer_ns();
      while (ld_relaxed_u64(p.bars) < target) {
        // an interval is microseconds; 10 s at a barrier means CTAs are missing (the launch did not fill the SMs the way
        // reserve_sms counts on, or somebody died): fail the launch rather than hang the device
        if (globaltimer_ns() - t_a > 10000000000ull) asm volatile("trap;");
      }
      __threadfence();
      t_b = globaltimer_ns();
      target += nb;
    }
    __syncthreads(); // the previous interval is complete everywhere
    for (uint32_t i = 0; i < P.done_n; i++) filter_final(p, P.done_b[i], P.done_ki[i], P.done_slot[i], gtid, gthreads);
    if (P.finished) break;
    if (planner) make_plan(&P, plans[(it + 1u) & 1u]);
    if (main_kind == MK_R0 && P.part == 0u && P.recal) {
      // every CTA published the rate of its round-0 passes (steps per time) a few streams ago: the shares of the stream
      // that begins are proportional to them.  Integer sums, so that every CTA derives the very same boundaries.
      unsigned long long tot = 0;
      // (up to gridDim.x >= nb: the entries beyond nb are zero.  Written with nb, ptxas (12.9) finds a worse register
      // allocation for the whole kernel -- 30 more bytes of spills in the hot loops, -4 % k-mer ops/s)
      for (uint32_t i = threadIdx.x; i < gridDim.x; i += blockDim.x) tot += __ldcg(p.speed + i);
      tot = block_sum(tot, red_sh[0]);
      const unsigned long long mean = max(1ull, tot / nb), lo = max(1ull, mean * 7ull / 10ull), hi = mean * 14ull / 10ull + 1ull;
      unsigned long long all = 0, before = 0, mine = 0;
      for (uint32_t i = threadIdx.x; i < nb; i += blockDim.x) {
        const unsigned long long v = min(max((unsigned long long)__ldcg(p.speed + i), lo), hi);
        all += v;
        if (i < bid) before += v;
        if (i == bid) mine = v;
      }
      all = block_sum(all, red_sh[0]); before = block_sum(before, red_sh[1]); mine = block_sum(mine, red_sh[2]);
      if (threadIdx.x <= uint32_t(kLevelWarps))
        cum_sh[P.cur.cum][threadIdx.x] = ((before * kLevelWarps + mine * threadIdx.x) << 32) / (all * kLevelWarps);
      __syncthreads();
    }

    for (uint32_t ph = 0; ph < 2u; ph++) {
      const bool tail_now = tail_on ? (tail_first ? ph == 0u : ph == 1u) : false;
      const bool main_now = tail_on ? !tail_now : ph == 0u;
      if (!tail_now && !(main_now && main_kind != MK_NONE)) continue;
      if (main_now && main_kind == MK_CLEAR) {
        for (uint64_t i = gtid; i < kCbfCounters * p.arrays; i += gthreads) p.V[i] = 0xFFFFFFFFu;
        continue;
      }
      if (main_now && main_kind == MK_R0) {
        // ---- round 0 (rows [row0, row1) of it): every occurrence writes its time into T_1 (the first toucher of a
        // counter wins) and goes to the warp's list, so that level 1 is an ordinary list round ----
        const uint32_t ki = P.cur.ki, batch = P.cur.batch, cb = P.cur.buf, n_steps = P.cur.n_steps;
        const uint64_t* cum = cum_sh[P.cur.cum] + wib;
        const StreamConsts sc = stream_consts(p.k[ki]);
        uint32_t* __restrict__ bf = p.bf_pool + (uint64_t(P.cur.slot) * p.nk + ki) * kBfWords;
        const SurvList lst = list_of(p, cb, n_steps, cum, gwarp_now);
        uint32_t cnt = P.part ? warp_cnt[cb][wib] : 0u;
        const uint32_t tag = P.cur.tag;
        uint32_t* __restrict__ VC = t1_array(P.cur);
        unsigned long long w_t0 = 0;
        uint32_t w_steps = 0;
        if (threadIdx.x == 0) w_t0 = globaltimer_ns();
        with_kmer_shape(sc, [&](auto shape) {
          for_runs<decltype(shape)::value>(p, c, cum, batch, ki, sc, n_steps, P.row0, P.row1,
                   [&](uint32_t s, uint32_t thr, bool valid, uint64_t h0, const uint32_t (&pw)[4]) {
                     const uint32_t t = s * 32u + c.lane;
                     const bool q = valid && thr > 0u;
                     if (q) {
#pragma unroll
                       for (int j = 0; j < 4; j++) red_min(VC + (pw[j] & 0xFFFFFFu), tag | t);
                       if (thr == 1u) bf_insert(bf, pw);
                     }
                     if (valid) ops++;
                     w_steps++;
                     surv_append(lst, cnt, q && thr > 1u, h0, t | (thr << kTimeBits), c.lane);
                   });
        });
        if (c.lane == 0) warp_cnt[cb][wib] = cnt;
        if (threadIdx.x == 0 && p.weighted) { cal_ns += globaltimer_ns() - w_t0; cal_steps += w_steps; }
        continue;
      }
      // ---- list round of the tail (level >= 2) or of the head (level 1) ----
      const StreamSt* S = tail_now ? &P.tail : &P.cur;
      const uint32_t sbuf = S->buf;
      const StreamConsts sc = stream_consts(p.k[S->ki]);
      ListJob J;
      J.L = S->L; J.lread = S->lread; J.tag = S->tag; J.tag_next = S->tag_next; J.vmask = vmask;
      J.lst = list_of(p, sbuf, S->n_steps, cum_sh[S->cum] + wib, gwarp_now);
      J.V = J.L == 1u ? t1_array(*S) : p.V + ((J.L + S->pb) & 1u) * kCbfCounters;
      J.Vn = p.V + ((J.L + 1u + S->pb) & 1u) * kCbfCounters;
      J.bf = p.bf_pool + (uint64_t(S->slot) * p.nk + S->ki) * kBfWords;
      J.cbf = p.cbf_pool ? p.cbf_pool + uint64_t(S->sid) * kCbfCounters : nullptr;
      J.cnt = warp_cnt[sbuf][wib];
      if (c.lane == 0) list_seen += J.cnt; // (diagnostic, flushed once at the end)
      if (pre_for != (tail_now ? 1u : 2u)) fetch_entries<2>(J.lst, J.cnt, 0, c.lane, nx_lo, nx_hi, nx_meta);
      pre_for = 0;
      const uint32_t kept = (J.cbf || J.L > 1u) ? list_round_all(J, sc, c.lane, nx_lo, nx_hi, nx_meta)
                                                 : list_round_first(J, sc, c.lane, nx_lo, nx_hi, nx_meta);
      __syncwarp();
      if (c.lane == 0) warp_cnt[sbuf][wib] = kept;
    }

    __syncthreads(); // every thread of the CTA has issued its part of the interval; the next plan is written
    if (threadIdx.x == 0) {
      const unsigned long long t_c = globaltimer_ns();
      if (main_kind == MK_R0 && P.publish && P.last_part && p.weighted) { // this CTA's round-0 rate, for the weighted shares
        p.speed[bid] = uint32_t(min(max(cal_steps * 4000000ull / max(cal_ns, 1ull), 1ull), 262143ull));
        cal_ns = 0; cal_steps = 0;
      }
      __threadfence();
      atomicAdd(p.bars, 1ull);
      // where the time of a CTA goes, per kind of interval: barrier wait, work, intervals (kept in shared memory:
      // global read-modify-writes here would make the reporting CTA late for every barrier)
      // 0 clear, 1 round 0 alone, 2 level-1 round alone, 3 late round alone, 4 round 0 + late round, 5 level-1 + late round
      const uint32_t kind = main_kind == MK_CLEAR ? 0u : main_kind == MK_R0 ? (tail_on ? 4u : 1u) : main_kind == MK_R1 ? (tail_on ? 5u : 2u) : 3u;
      diag[kind * 3 + 0] += t_b - t_a;
      diag[kind * 3 + 1] += t_c - t_b;
      diag[kind * 3 + 2] += 1;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ops += __shfl_xor_sync(0xffffffffu, ops, o);
  if (c.lane == 0 && ops) atomicAdd(p.counters + 0, ops);
  if (c.lane == 0 && list_seen) atomicAdd(p.counters + 17, list_seen);
  if (bid == 0 && threadIdx.x == 0) atomicMax(p.counters + 21, globaltimer_ns());
  if (bid == p.report_cta && threadIdx.x == 0)
    for (uint32_t i = 0; i < kLevelDiag; i++) p.counters[kLevelDiagAt + i] += diag[i]; // several waves add up
  if (p.cta_times && threadIdx.x < kLevelDiag) p.cta_times[bid * 32u + threadIdx.x] = diag[threadIdx.x];
#undef bid
#undef nb
#undef gtid
#undef gthreads
#undef gwarp_now
}

// ---- known-answer support: the hashes exactly as the build kernels compute them ----
// Every k-mer start of one uploaded read through the device's own path (packed words + mask window, shared-memory byte
// tables, hash_h0, the multiply-xorshift extra hashes): h[4 * pos .. 4 * pos + 3] and valid[pos] for pos < npos.
__global__ void __launch_bounds__(kLevelWarps * 32) debug_nthash_kernel(const uint64_t* __restrict__ pk, const uint32_t* __restrict__ nm,
                                                                        uint64_t wbase, uint32_t len, uint32_t k,
                                                                        uint64_t* __restrict__ h, uint8_t* __restrict__ valid)
{
  __shared__ uint64_t tf[8 * 256];
  __shared__ uint64_t tr[8 * 256];
  fill_hash_tables(tf, tr);
  __syncthreads();
  if (len < k) return;
  const StreamConsts sc = stream_consts(k);
  const uint32_t npos = len - k + 1, lane = threadIdx.x & 31u;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  with_kmer_shape(sc, [&](auto shape) {
    for (uint32_t s = warp; s * 32u < npos; s += nwarps) {
      const uint64_t w0 = __ldg(pk + wbase + s), w1 = __ldg(pk + wbase + s + 1);
      const uint32_t m0 = __ldg(nm + wbase + s), m1 = __ldg(nm + wbase + s + 1);
      uint64_t h0 = 0;
      const bool ok = hash_h0<decltype(shape)::value>(tf, tr, w0, w1, m0, m1, s * 32u, npos, lane, sc, h0);
      const uint32_t pos = s * 32u + lane;
      if (pos < npos) {
        valid[pos] = ok ? 1 : 0;
        uint64_t h1 = h0 * sc.mul1, h2 = h0 * sc.mul2, h3 = h0 * sc.mul3;
        h1 ^= h1 >> kMultiShift; h2 ^= h2 >> kMultiShift; h3 ^= h3 >> kMultiShift;
        h[4 * uint64_t(pos) + 0] = ok ? h0 : 0; h[4 * uint64_t(pos) + 1] = ok ? h1 : 0;
        h[4 * uint64_t(pos) + 2] = ok ? h2 : 0; h[4 * uint64_t(pos) + 3] = ok ? h3 : 0;
      }
    }
  });
}

void launch_debug_nthash(const uint64_t* pk, const uint32_t* nm, uint64_t wbase, uint32_t len, uint32_t k, uint64_t* h,
                         uint8_t* valid, cudaStream_t s)
{
  debug_nthash_kernel<<<8, kLevelWarps * 32, 0, s>>>(pk, nm, wbase, len, k, h, valid);
}

int levels_ctas_per_sm(int ctas_per_sm)
{
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, build_filters_levels_kernel, kLevelWarps * 32, 0);
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  if (ctas_per_sm > 0) per_sm = std::min(per_sm, ctas_per_sm);
  if (const char* e = std::getenv("GP_LEVEL_CTAS")) per_sm = std::max(1, std::min(per_sm, std::atoi(e))); // experiments
  return per_sm;
}

int levels_max_grid(int sm_count, int ctas_per_sm) { return sm_count * levels_ctas_per_sm(ctas_per_sm); }

void preload_levels()
{
  cudaFuncAttributes a;
  if (cudaFuncGetAttributes(&a, (const void*)build_filters_levels_kernel) != cudaSuccess) cudaGetLastError();
  if (cudaFuncGetAttributes(&a, (const void*)fill_anchor_kernel) != cudaSuccess) cudaGetLastError();
}

cudaError_t launch_build_filters_levels(const LevelParams& p, int sm_count, cudaStream_t s, int ctas_per_sm)
{
  if (p.n_streams == 0) return cudaSuccess;
  // 132 KB of shared memory (3 CTAs x 33 KB), the rest L1; the edit kernel asks for the same so that the two can
  // share an SM.  Function attributes are per device: set on every launch (a cheap host-side call).
  cudaFuncSetAttribute((const void*)build_filters_levels_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 58);
  LevelParams lp = p;
  lp.sms = uint32_t(sm_count);
  if (lp.keep_sms == 0 || lp.keep_sms > lp.sms || !lp.sm_table) lp.keep_sms = lp.sms; // every SM builds
  lp.n_ctas = lp.keep_sms * uint32_t(levels_ctas_per_sm(ctas_per_sm));
  void* args[] = { &lp };
  // cooperative launch: the barriers need every CTA resident
  return cudaLaunchCooperativeKernel((const void*)build_filters_levels_kernel, dim3(sm_count * levels_ctas_per_sm(ctas_per_sm)),
                                     dim3(kLevelWarps * 32), args, 0, s);
}

} // namespace gp
