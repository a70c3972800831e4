// Read packing and the counting-Bloom-gated Bloom filter build (sm_100a).
//
// Replaces fill_bfs (bcgsc/goldpolish src/utils.cpp:96-123) and the per-batch loop around it
// (src/goldpolish_targeted_bfs.cpp:124-140).  One warp owns one (batch, k) stream and walks it
// in the reference's order -- reads as listed, positions ascending -- 32 k-mers per step.
// Inside a step the warp keeps the reference's sequential semantics exactly:
//   * lanes whose four counters are touched by no lower lane of the step ("independent")
//     read-modify-write in parallel: their result cannot depend on any other lane;
//   * the remaining lanes (same k-mer twice in 32 positions, or a chance counter collision)
//     are replayed one at a time in lane order against the updated counters.
// Bloom-filter bit sets commute, so they are plain 32-bit atomicOr.
#include "gp_common.cuh"
#include "gp_kernels.cuh"
#include "gp_hashing.cuh"

#include <cstdio>
#include <cstdlib>

namespace gp {

// ------------------------------------------------------------------------------------
// pack: ASCII -> 2 bits/base (32 bases per u64) + 1 bit/base "no seed" mask (32 per u32)
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) pack_reads_kernel(const char* __restrict__ ascii,
                                                         const uint64_t* __restrict__ ascii_off,
                                                         const uint64_t* __restrict__ base_off, // multiple of 32
                                                         uint64_t* __restrict__ pk, uint32_t* __restrict__ nm,
                                                         uint32_t n_reads)
{
  for (uint32_t r = blockIdx.x; r < n_reads; r += gridDim.x) {
    const uint64_t a0 = ascii_off[r];
    const uint32_t len = uint32_t(ascii_off[r + 1] - a0);
    const uint64_t g0 = base_off[r] >> 5;
    const uint32_t groups = (len + 31u) >> 5;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(ascii) + a0;
    for (uint32_t gi = threadIdx.x; gi < groups; gi += blockDim.x) {
      uint64_t w = 0;
      uint32_t m = 0;
      const uint32_t base = gi << 5;
#pragma unroll 8
      for (uint32_t i = 0; i < 32; i++) {
        const uint32_t q = base + i;
        uint32_t c = q < len ? src[q] : 0u;
        const uint32_t lc = c | 0x20u;
        const bool ok = (lc == 'a') | (lc == 'c') | (lc == 'g') | (lc == 't');
        uint32_t x = (lc >> 1) & 3u; // a:0 c:1 g:3 t:2
        x ^= x >> 1;                 // a:0 c:1 g:2 t:3
        w |= uint64_t(ok ? x : 0u) << (2 * i);
        m |= (ok ? 0u : 1u) << i;
      }
      pk[g0 + gi] = w;
      nm[g0 + gi] = m;
    }
  }
}

void launch_pack_reads(const char* ascii, const uint64_t* ascii_off, const uint64_t* base_off, uint64_t* pk,
                       uint32_t* nm, uint32_t n_reads, cudaStream_t s)
{
  if (n_reads == 0) return;
  const uint32_t grid = n_reads < 148u * 16u ? n_reads : 148u * 16u;
  pack_reads_kernel<<<grid, 128, 0, s>>>(ascii, ascii_off, base_off, pk, nm, n_reads);
}

// ------------------------------------------------------------------------------------
// build
// ------------------------------------------------------------------------------------
constexpr int kBuildWarps = 8;
constexpr int kTabBits = 9;
constexpr int kTabSlots = 1 << kTabBits;
constexpr size_t kBuildSmem = 2 * 8 * 256 * sizeof(uint64_t) + size_t(kBuildWarps) * kTabSlots * sizeof(uint32_t);

__device__ __forceinline__ void cbf_bf_apply(uint8_t* __restrict__ cbf, uint32_t* __restrict__ bf,
                                             const uint32_t (&ci)[4], const uint32_t (&bi)[4],
                                             const uint32_t (&c)[4], uint32_t thr)
{
  const uint32_t mn = min(min(c[0], c[1]), min(c[2], c[3]));
  uint32_t cnt = mn;
  if (mn < thr) {
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (c[j] == mn) __stcg(cbf + ci[j], (uint8_t)(mn + 1));
    cnt = mn + 1;
  }
  if (cnt >= thr) {
#pragma unroll
    for (int j = 0; j < 4; j++) atomicOr(bf + (bi[j] >> 5), 1u << (bi[j] & 31u));
  }
}

// ---- pieces shared by the two build kernels -------------------------------------------------

// Per-lane registers that hold 32 consecutive packed / mask words of the current read (one word
// per lane) and the 32 that follow.  Every read starts on a word boundary, so step s (32 k-mer
// starts) needs words s and s+1 -- the same for all lanes: they are handed out by shuffle, and
// the look-ahead registers are only touched on the last step of a chunk, 31 steps after their load.
__device__ __forceinline__ void seq_load_chunk(const BuildParams& p, uint64_t wbase, uint32_t nwords, uint32_t chunk,
                                               uint32_t lane, uint64_t& pkw, uint32_t& nmw)
{
  const uint32_t wq = chunk * 32u + lane;
  const bool in = wq <= nwords; // one spare word is always allocated behind a read
  pkw = in ? __ldg(p.pk + wbase + wq) : 0ull;
  nmw = in ? __ldg(p.nm + wbase + wq) : 0xFFFFFFFFu;
}

// Commit one step in stream order.  `c` holds the counters loaded for the valid lanes.
// Which lanes share a counter with a LOWER lane of this step?  Lanes publish themselves in a
// small direct-mapped table of lane masks (slot = hash of the counter index); slot sharing only
// nominates candidates, the counter indices themselves are then compared through shuffles, so
// the answer is exact whatever the table size.  Independent lanes update in parallel, the rest
// are replayed one at a time in lane order against the updated counters.
__device__ __forceinline__ void commit_step(uint8_t* __restrict__ cbf, uint32_t* __restrict__ bf, uint32_t* tab,
                                            uint32_t lane, bool valid, const uint32_t (&ci)[4], const uint32_t (&bi)[4],
                                            uint32_t (&c)[4], uint32_t thr, unsigned long long& ops,
                                            unsigned long long& serial)
{
  uint32_t sl[4];
  if (valid) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      sl[j] = (ci[j] * 2654435761u) >> (32 - kTabBits);
      atomicOr(&tab[sl[j]], 1u << lane);
    }
  }
  __syncwarp();
  uint32_t lower = 0;
  if (valid) {
#pragma unroll
    for (int j = 0; j < 4; j++) lower |= tab[sl[j]];
    lower &= (1u << lane) - 1u;
  }
  __syncwarp();
  if (valid) {
#pragma unroll
    for (int j = 0; j < 4; j++) tab[sl[j]] = 0u; // leave the table clean for the next step
  }
  bool indep = true;
  const uint32_t rounds = __reduce_max_sync(0xffffffffu, (uint32_t)__popc(lower));
  for (uint32_t it = 0; it < rounds; it++) {
    const uint32_t l = lower ? (uint32_t)__ffs(lower) - 1u : lane;
    lower &= lower - 1u;
    const uint32_t o0 = __shfl_sync(0xffffffffu, ci[0], l), o1 = __shfl_sync(0xffffffffu, ci[1], l);
    const uint32_t o2 = __shfl_sync(0xffffffffu, ci[2], l), o3 = __shfl_sync(0xffffffffu, ci[3], l);
    if (l != lane) {
#pragma unroll
      for (int j = 0; j < 4; j++) indep &= (ci[j] != o0) & (ci[j] != o1) & (ci[j] != o2) & (ci[j] != o3);
    }
  }
  if (valid) {
    if (indep) cbf_bf_apply(cbf, bf, ci, bi, c, thr);
    ops++;
  }
  uint32_t dep = __ballot_sync(0xffffffffu, valid && !indep);
  while (dep) {
    __syncwarp();
    const uint32_t l = __ffs(dep) - 1;
    if (lane == l) {
#pragma unroll
      for (int j = 0; j < 4; j++) c[j] = __ldcg(cbf + ci[j]);
      cbf_bf_apply(cbf, bf, ci, bi, c, thr);
      serial++;
    }
    dep &= dep - 1;
  }
  __syncwarp(); // orders this step's counter stores before the next step's loads
}

__device__ __forceinline__ void flush_counters(const BuildParams& p, uint32_t lane, unsigned long long ops,
                                               unsigned long long serial)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ops += __shfl_xor_sync(0xffffffffu, ops, o);
    serial += __shfl_xor_sync(0xffffffffu, serial, o);
  }
  if (lane == 0) {
    if (ops) atomicAdd(p.counters + 0, ops);
    if (serial) atomicAdd(p.counters + 1, serial);
  }
}

// ---- one warp per stream --------------------------------------------------------------------
// Steps are software-pipelined: while step i waits for its counters, step i+1 is already hashed
// and its counter sectors are prefetched into L2.  Loads of step i+1 are only ISSUED after step
// i has stored.  Define GP_BUILD_TIMING to print the per-phase cycle budget of long streams.
#ifndef GP_BUILD_MIN_CTAS
#define GP_BUILD_MIN_CTAS 3
#endif
__global__ void __launch_bounds__(kBuildWarps * 32, GP_BUILD_MIN_CTAS) build_filters_kernel(BuildParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* tf = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* tr = tf + 8 * 256;
  uint32_t* tabs = reinterpret_cast<uint32_t*>(tr + 8 * 256);
  fill_hash_tables(tf, tr);
  for (uint32_t i = threadIdx.x; i < (blockDim.x >> 5) * kTabSlots; i += blockDim.x) tabs[i] = 0u;
  __syncthreads();

  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp = threadIdx.x >> 5;
  uint32_t* tab = tabs + warp * kTabSlots;
  unsigned long long ops = 0, serial = 0;
#ifdef GP_BUILD_TIMING
  long long tim[4] = { 0, 0, 0, 0 };
#endif

  for (;;) {
    uint32_t slot = 0;
    if (lane == 0) slot = atomicAdd(p.next_stream, 1u);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    if (slot >= p.n_streams) break;
    const uint32_t sid = p.stream_order[slot]; // local stream id within this wave
    const uint32_t lb = sid / p.nk, ki = sid - lb * p.nk;
    const uint32_t batch = p.first_batch + lb;
    const StreamConsts sc = stream_consts(p.k[ki]);
    uint8_t* __restrict__ cbf = p.cbf_pool + uint64_t(sid) * kCbfCounters;
    uint32_t* __restrict__ bf = p.bf_pool + (uint64_t(p.bf_slot ? p.bf_slot[batch] : batch) * p.nk + ki) * kBfWords;

    const uint64_t e0 = p.batch_entry_off[batch], e1 = p.batch_entry_off[batch + 1];
    with_kmer_shape(sc, [&](auto shape) {
      constexpr bool PARTIAL = decltype(shape)::value;
      for (uint64_t e = e0; e < e1; e++) {
        const gp_read_entry ent = p.entries[e];
        const uint32_t thr = ent.kmer_threshold - 2u + ki; // utils.cpp:108,121
        const uint32_t len = p.read_len[ent.read_id];
        if (len < sc.k) continue;
        const uint64_t wbase = p.read_boff[ent.read_id] >> 5;
        const uint32_t npos = len - sc.k + 1;
        const uint32_t nwords = (len + 31u) >> 5;
        SeqRegs sr;
        seq_load_chunk(p, wbase, nwords, 0, lane, sr.pk_cur, sr.nm_cur);
        seq_load_chunk(p, wbase, nwords, 1, lane, sr.pk_nxt, sr.nm_nxt);
        uint32_t ci[4], bi[4], c[4], nci[4], nbi[4];
        bool valid = hash_step<PARTIAL>(tf, tr, sr, 0, 0, npos, lane, sc, ci, bi), nvalid = false;
        if (valid) {
#pragma unroll
          for (int j = 0; j < 4; j++) c[j] = __ldcg(cbf + ci[j]);
        }
        for (uint32_t p0 = 0, step = 0; p0 < npos; p0 += 32, step++) {
          const bool has_next = p0 + 32 < npos;
#ifdef GP_BUILD_TIMING
          const long long tA = clock64();
#endif
          if (has_next) {
            if (((step + 1) & 31u) == 0u) { // entering the next chunk of 32 steps
              sr.pk_cur = sr.pk_nxt; sr.nm_cur = sr.nm_nxt;
              seq_load_chunk(p, wbase, nwords, ((step + 1) >> 5) + 1, lane, sr.pk_nxt, sr.nm_nxt);
            }
            nvalid = hash_step<PARTIAL>(tf, tr, sr, step + 1, p0 + 32, npos, lane, sc, nci, nbi);
            if (nvalid) {
#pragma unroll
              for (int j = 0; j < 4; j++) asm volatile("prefetch.global.L2 [%0];" ::"l"(cbf + nci[j]));
            }
          }
#ifdef GP_BUILD_TIMING
          const long long tB = clock64();
#endif
          commit_step(cbf, bf, tab, lane, valid, ci, bi, c, thr, ops, serial);
#ifdef GP_BUILD_TIMING
          const long long tC = clock64();
          tim[0] += tB - tA; tim[1] += tC - tB; tim[2]++;
#endif
          if (has_next) {
            valid = nvalid;
#pragma unroll
            for (int j = 0; j < 4; j++) { ci[j] = nci[j]; bi[j] = nbi[j]; }
            if (valid) {
#pragma unroll
              for (int j = 0; j < 4; j++) c[j] = __ldcg(cbf + ci[j]);
            }
          }
        }
      }
    });
  }
#ifdef GP_BUILD_TIMING
  if (lane == 0 && tim[2] > 1000)
    printf("warp: %lld steps, hash %lld + commit %lld cycles/step\n", tim[2], tim[0] / tim[2], tim[1] / tim[2]);
#endif
  flush_counters(p, lane, ops, serial);
}

// ---- one HASH warp and one COMMIT warp per stream ---------------------------------------------
// A lone stream is bound by the length of one warp's dependent instruction chain per step, not
// by memory.  Splitting the step shortens that chain: the hash warp extracts, hashes, derives
// the indices of 32 k-mers, prefetches the counter sectors into L2 and hands the indices over
// through a shared-memory ring; the commit warp only loads, resolves intra-step sharing and
// updates -- in stream order, exactly as build_filters_kernel does.
constexpr int kPairs = 4;            // pairs per CTA (8 warps)
constexpr int kRingDepth = 2;        // steps in flight between the two warps of a pair
constexpr uint32_t kMsgStep = 0, kMsgBegin = 1, kMsgQuit = 2;

struct PairSlot {
  uint32_t type, valid_mask, thr, sid, batch, ki, pad0, pad1;
  uint32_t ci[4][32];
  uint32_t bi[4][32];
};
struct PairRing {
  PairSlot slot[kRingDepth];
  volatile uint32_t head, tail; // produced / consumed message counts
  uint32_t pad[6];
};
constexpr size_t kPairSmem = 2 * 8 * 256 * sizeof(uint64_t) + size_t(kPairs) * kTabSlots * sizeof(uint32_t) +
                             size_t(kPairs) * sizeof(PairRing);

__device__ __forceinline__ PairSlot* ring_acquire(PairRing* r, uint32_t head)
{ // producer: wait for a free slot
  while (head - r->tail >= uint32_t(kRingDepth)) { }
  return &r->slot[head % kRingDepth];
}
__device__ __forceinline__ void ring_publish(PairRing* r, uint32_t& head, uint32_t lane)
{
  // data and flag live in the same SM's shared memory, written in program order by one warp;
  // __syncwarp orders the lanes' slot stores before lane 0 raises the flag.  (A CTA-scope
  // membar here would also wait for this warp's outstanding global prefetches.)
  __syncwarp();
  head++;
  if (lane == 0) r->head = head;
}

__global__ void __launch_bounds__(kPairs * 64) build_filters_paired_kernel(BuildParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* tf = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* tr = tf + 8 * 256;
  uint32_t* tabs = reinterpret_cast<uint32_t*>(tr + 8 * 256);
  PairRing* rings = reinterpret_cast<PairRing*>(tabs + kPairs * kTabSlots);
  fill_hash_tables(tf, tr);
  for (uint32_t i = threadIdx.x; i < kPairs * kTabSlots; i += blockDim.x) tabs[i] = 0u;
  if (threadIdx.x < kPairs) { rings[threadIdx.x].head = 0; rings[threadIdx.x].tail = 0; }
  __syncthreads();

  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t pair = warp >> 1;
  PairRing* ring = rings + pair;

  if ((warp & 1u) == 0u) {
    // ------------------------------- hash warp -------------------------------
    uint32_t head = 0;
    for (;;) {
      uint32_t qslot = 0;
      if (lane == 0) qslot = atomicAdd(p.next_stream, 1u);
      qslot = __shfl_sync(0xffffffffu, qslot, 0);
      if (qslot >= p.n_streams) break;
      const uint32_t sid = p.stream_order[qslot];
      const uint32_t lb = sid / p.nk, ki = sid - lb * p.nk;
      const uint32_t batch = p.first_batch + lb;
      const StreamConsts sc = stream_consts(p.k[ki]);
      const uint8_t* cbf = p.cbf_pool + uint64_t(sid) * kCbfCounters;
      {
        PairSlot* sl = ring_acquire(ring, head);
        if (lane == 0) { sl->type = kMsgBegin; sl->sid = sid; sl->batch = batch; sl->ki = ki; }
        ring_publish(ring, head, lane);
      }
      const uint64_t e0 = p.batch_entry_off[batch], e1 = p.batch_entry_off[batch + 1];
      with_kmer_shape(sc, [&](auto shape) {
        constexpr bool PARTIAL = decltype(shape)::value;
        for (uint64_t e = e0; e < e1; e++) {
          const gp_read_entry ent = p.entries[e];
          const uint32_t thr = ent.kmer_threshold - 2u + ki; // utils.cpp:108,121
          const uint32_t len = p.read_len[ent.read_id];
          if (len < sc.k) continue;
          const uint64_t wbase = p.read_boff[ent.read_id] >> 5;
          const uint32_t npos = len - sc.k + 1;
          const uint32_t nwords = (len + 31u) >> 5;
          SeqRegs sr;
          seq_load_chunk(p, wbase, nwords, 0, lane, sr.pk_cur, sr.nm_cur);
          seq_load_chunk(p, wbase, nwords, 1, lane, sr.pk_nxt, sr.nm_nxt);
          for (uint32_t p0 = 0, step = 0; p0 < npos; p0 += 32, step++) {
            if (step && (step & 31u) == 0u) {
              sr.pk_cur = sr.pk_nxt; sr.nm_cur = sr.nm_nxt;
              seq_load_chunk(p, wbase, nwords, (step >> 5) + 1, lane, sr.pk_nxt, sr.nm_nxt);
            }
            uint32_t ci[4], bi[4];
            const bool valid = hash_step<PARTIAL>(tf, tr, sr, step, p0, npos, lane, sc, ci, bi);
            if (valid) {
#pragma unroll
              for (int j = 0; j < 4; j++) asm volatile("prefetch.global.L2 [%0];" ::"l"(cbf + ci[j]));
            }
            const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
            if (vmask == 0u) continue; // nothing to commit in this step
            PairSlot* sl = ring_acquire(ring, head);
#pragma unroll
            for (int j = 0; j < 4; j++) { sl->ci[j][lane] = ci[j]; sl->bi[j][lane] = bi[j]; }
            if (lane == 0) { sl->type = kMsgStep; sl->valid_mask = vmask; sl->thr = thr; }
            ring_publish(ring, head, lane);
          }
        }
      });
    }
    PairSlot* sl = ring_acquire(ring, head);
    if (lane == 0) sl->type = kMsgQuit;
    ring_publish(ring, head, lane);
    return;
  }

  // ------------------------------- commit warp -------------------------------
  uint32_t* tab = tabs + pair * kTabSlots;
  unsigned long long ops = 0, serial = 0;
  uint32_t tail = 0;
  uint8_t* cbf = nullptr;
  uint32_t* bf = nullptr;
  for (;;) {
    while (ring->head == tail) { }
    __syncwarp();
    const volatile PairSlot* sl = &ring->slot[tail % kRingDepth];
    const uint32_t type = sl->type;
    if (type == kMsgQuit) break;
    if (type == kMsgBegin) {
      cbf = p.cbf_pool + uint64_t(sl->sid) * kCbfCounters;
      bf = p.bf_pool + (uint64_t(p.bf_slot ? p.bf_slot[sl->batch] : sl->batch) * p.nk + sl->ki) * kBfWords;
      __syncwarp();
      tail++;
      if (lane == 0) ring->tail = tail;
      continue;
    }
    const uint32_t vmask = sl->valid_mask, thr = sl->thr;
    uint32_t ci[4], bi[4], c[4];
#pragma unroll
    for (int j = 0; j < 4; j++) { ci[j] = sl->ci[j][lane]; bi[j] = sl->bi[j][lane]; }
    __syncwarp();
    tail++;
    if (lane == 0) ring->tail = tail; // the hash warp may reuse the slot
    const bool valid = (vmask >> lane) & 1u;
    if (valid) {
#pragma unroll
      for (int j = 0; j < 4; j++) c[j] = __ldcg(cbf + ci[j]);
    }
    commit_step(cbf, bf, tab, lane, valid, ci, bi, c, thr, ops, serial);
  }
  flush_counters(p, lane, ops, serial);
}

void launch_build_filters(const BuildParams& p, int sm_count, cudaStream_t s)
{
  if (p.n_streams == 0) return;
  static bool configured = false;
  if (!configured) {
    cudaFuncSetAttribute(build_filters_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kBuildSmem));
    cudaFuncSetAttribute(build_filters_paired_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kPairSmem));
    configured = true;
  }
  // One warp per stream.  With few streams the CTAs are made small so that the warps spread over
  // all SMs (a lone warp per SM runs a step noticeably faster than eight sharing one SM).
  uint32_t warps = kBuildWarps;
  if (p.n_streams < uint32_t(sm_count) * kBuildWarps) {
    warps = (p.n_streams + uint32_t(sm_count) - 1) / uint32_t(sm_count);
    if (warps < 1) warps = 1;
    if (warps > uint32_t(kBuildWarps)) warps = kBuildWarps;
  }
  bool paired = false; // the paired kernel is kept for experiments: GP_BUILD_KERNEL=p
  if (const char* f = std::getenv("GP_BUILD_KERNEL")) paired = f[0] == 'p';
  if (paired) {
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, build_filters_paired_kernel, kPairs * 64, kPairSmem);
    if (per_sm < 1) per_sm = 1;
    uint32_t grid = uint32_t(sm_count) * uint32_t(per_sm);
    const uint32_t need = (p.n_streams + kPairs - 1) / kPairs;
    if (grid > need) grid = need;
    build_filters_paired_kernel<<<grid, kPairs * 64, kPairSmem, s>>>(p);
    return;
  }
  const size_t smem = 2 * 8 * 256 * sizeof(uint64_t) + size_t(warps) * kTabSlots * sizeof(uint32_t);
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, build_filters_kernel, int(warps * 32), smem);
  if (per_sm < 1) per_sm = 1;
  uint32_t grid = uint32_t(sm_count) * uint32_t(per_sm);
  const uint32_t need = (p.n_streams + warps - 1) / warps;
  if (grid > need) grid = need;
  build_filters_kernel<<<grid, warps * 32, smem, s>>>(p);
}

// ------------------------------------------------------------------------------------
// random-access roof: the build kernel's memory shape with the hashing taken out
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) roof_kernel(uint8_t* cbf_pool, uint32_t* bf_pool, uint64_t region,
                                                   uint32_t iters, uint32_t total_warps, int mode)
{
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (gw >= total_warps) return;
  uint8_t* cbf = cbf_pool + uint64_t(gw) * region;
  uint32_t* bf = bf_pool + uint64_t(gw) * kBfWords;
  uint64_t x = 0x9e3779b97f4a7c15ULL * (uint64_t(gw) * 32 + lane + 1);
  if (mode >= 3) {
    // (mode 4: atomicMin rounds only, mode 5: load rounds only)
    // the level-synchronous kernel's shape: ALL warps share one array of 32-bit timestamps the
    // size of one counting filter (40 MiB, L2 resident); a round is 4 atomicMin, the next 4 loads
    uint32_t* V = reinterpret_cast<uint32_t*>(cbf_pool);
    uint32_t acc = 0;
    for (uint32_t it = 0; it < iters; it++) {
      uint32_t ci[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        ci[j] = uint32_t((x >> 11) % kCbfCounters);
      }
      if (mode == 4 || (mode == 3 && (it & 1u) == 0u)) {
#pragma unroll
        for (int j = 0; j < 4; j++) atomicMin(V + ci[j], uint32_t(x >> 32) | (it << 26));
      } else {
#pragma unroll
        for (int j = 0; j < 4; j++) acc ^= __ldcg(V + ci[j]);
      }
    }
    if (acc == 0x12345678u) bf[0] = acc;
    return;
  }
  for (uint32_t it = 0; it < iters; it++) {
    uint32_t ci[4], bi[4], c[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      x ^= x << 13; x ^= x >> 7; x ^= x << 17;
      ci[j] = uint32_t((x >> 11) % region);
      bi[j] = uint32_t(x) & uint32_t(kBfBits - 1);
    }
#pragma unroll
    for (int j = 0; j < 4; j++) c[j] = __ldcg(cbf + ci[j]);
    const uint32_t mn = min(min(c[0], c[1]), min(c[2], c[3]));
    // alternate between the two halves of the algorithmic traffic: counter write-back below
    // the threshold, filter bit sets at it
    if (mode == 1) { // loads only (experiment)
      if (mn == 255u) bf[0] = 1u;
    } else if ((it & 1u) == 0u || mode == 2) {
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (c[j] == mn) __stcg(cbf + ci[j], (uint8_t)((mn + 1) & 15u));
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) atomicOr(bf + (bi[j] >> 5), 1u << (bi[j] & 31u));
    }
    __syncwarp();
  }
}

void launch_roof(uint8_t* cbf_pool, uint32_t* bf_pool, uint64_t region, uint32_t iters, uint32_t warps, cudaStream_t s)
{
  const uint32_t threads = 256;
  const uint32_t grid = (warps * 32 + threads - 1) / threads;
  // 0: the warp-per-stream kernel's mix (private 10 MiB regions); 3: the level-synchronous kernel's
  // shape (one shared 40 MiB array in L2); GP_ROOF_MODE=1 loads only, 2 loads + counter stores
  int mode = 0;
  if (const char* m = std::getenv("GP_ROOF_MODE")) mode = std::atoi(m);
  roof_kernel<<<grid, threads, 0, s>>>(cbf_pool, bf_pool, region, iters, warps, mode);
}

} // namespace gp
