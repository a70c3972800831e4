// k-mer support (gp_polish_fetch_support): how many k-mers of the draft and of the polished record of every contig the
// filters of its batch contain, for every k of the chain; and how many bits every (batch, k) filter has set.  See
// include/goldpolish_b200.h for the counting rule and DESIGN §4.7 for the shape.
//
// Both records of every contig of a launch are indexed by STEPS of 32 positions: record 2 i is the draft of contig i of
// the launch, record 2 i + 1 its polished record (no steps when it was dropped).  One inclusive scan of the steps per
// record gives the flattened index; every warp takes an equal run of it, whatever the record lengths.  A step reads its
// 64 bytes as two coalesced byte loads per lane, turns them into the 2-bit words and "no seed" masks of the packed read
// store with ballots, and hashes the 32 k-mers that start in it for every k with the build kernels' hash_from_words
// (4 bases per table lookup).  Counts are reduced per warp with ballots and kept per warp in shared memory until the
// warp's run leaves the record; then one atomic per (record, k) adds them.  The warp also stores the step's
// unsupported starts (valid and not present, one ballot word per k) into a bitmap addressed per contig (SupportMiss),
// which outlives the filters.
//
// Unsupported runs (gp_polish_fetch_unsupported) come from that bitmap, once per polish: the words of every (contig,
// record, k) form one flat range, a thread per word.  With miss(q) the bit of start q, a position is covered when
// miss(q - d) for some d < k <= 32, so the coverage of a word follows from the word and the one before it; a run starts
// at a covered position after an uncovered one and ends at a covered position before an uncovered one (the next word's
// first bit decides for bit 31).  One scan of the run starts numbers the runs; one of the miss popcounts makes a run's
// kmers the difference of two prefix values.
#include "gp_kernels.cuh"
#include "gp_hashing.cuh"

#include <cub/device/device_scan.cuh>

#include <algorithm>

namespace gp {

namespace {

constexpr int kSupportWarps = 8;

__device__ __forceinline__ uint32_t contig_of_launch(const SupportInput& in, uint32_t i) { return in.ids ? in.ids[i] : i; }

// record r of the launch: its bytes and length (a polished record is read no further than its buffer)
__device__ __forceinline__ const char* record_of(const SupportInput& in, uint32_t r, uint32_t& len)
{
  const uint32_t c = contig_of_launch(in, r >> 1);
  if (!(r & 1u)) {
    const uint64_t d0 = in.draft_off[c];
    len = uint32_t(in.draft_off[c + 1] - d0);
    return in.draft + d0;
  }
  const uint64_t c0 = in.cap_off[c];
  len = in.dropped[c] ? 0u : min(in.len[c], uint32_t(in.cap_off[c + 1] - c0));
  return in.buf[in.which[c]] + c0;
}

__global__ void support_steps_kernel(SupportInput in, uint32_t kmin, uint64_t* __restrict__ steps)
{
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < 2 * in.n; r += gridDim.x * blockDim.x) {
    uint32_t len;
    record_of(in, r, len);
    steps[r] = len >= kmin ? (uint64_t(len) + 31u) >> 5 : 0u;
  }
}

// 32 bits spread to the even bits of a word
__device__ __forceinline__ uint64_t spread_bits(uint32_t x)
{
  uint64_t v = x;
  v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
  v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
  v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
  v = (v | (v << 2)) & 0x3333333333333333ull;
  v = (v | (v << 1)) & 0x5555555555555555ull;
  return v;
}

// positions p .. p + 31 of a record as the packed read store holds them (pack_reads_kernel): 2-bit codes a:0 c:1 g:2 t:3
// of either case, and a mask bit for every other byte and every position past the end
__device__ __forceinline__ void pack_32(const char* rec, uint32_t len, uint32_t p, uint32_t lane, uint64_t& w, uint32_t& m)
{
  const uint32_t q = p + lane;
  const uint32_t lc = (q < len ? uint32_t((unsigned char)rec[q]) : 0u) | 0x20u;
  const bool ok = (lc == 'a') | (lc == 'c') | (lc == 'g') | (lc == 't');
  uint32_t x = (lc >> 1) & 3u;
  x ^= x >> 1;
  x = ok ? x : 0u;
  m = ~__ballot_sync(0xffffffffu, ok);
  w = spread_bits(__ballot_sync(0xffffffffu, x & 1u)) | (spread_bits(__ballot_sync(0xffffffffu, x & 2u)) << 1);
}

// first bitmap word of record r (0 draft, 1 polished) of contig c for k index j (layout: SupportMiss)
__device__ __forceinline__ uint64_t miss_base(const uint64_t* draft_off, const uint64_t* cap_off, uint64_t draft_words,
                                              uint64_t polished_words, uint32_t nk, uint32_t c, uint32_t r, uint32_t j)
{
  return r ? uint64_t(nk) * draft_words + uint64_t(j) * polished_words + (cap_off[c] >> 5) + c
           : uint64_t(j) * draft_words + (draft_off[c] >> 5) + c;
}

__global__ void __launch_bounds__(kSupportWarps * 32) support_count_kernel(SupportInput in, const uint64_t* __restrict__ step_end,
                                                                            SupportMiss miss)
{
  __shared__ uint64_t tf[8 * 256];
  __shared__ uint64_t tr[8 * 256];
  __shared__ uint32_t acc[kSupportWarps][kMaxK][2];
  fill_hash_tables(tf, tr);
  __syncthreads();
  if (*in.error || in.n == 0) return; // an unfinished polish: it runs again, and so does this
  const uint32_t lane = threadIdx.x & 31u, wib = threadIdx.x >> 5;
  const uint64_t warp = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5, nwarps = (uint64_t(gridDim.x) * blockDim.x) >> 5;
  const uint32_t n_rec = 2 * in.n;
  const uint64_t total = step_end[n_rec - 1];
  const uint64_t per = (total + nwarps - 1) / nwarps;
  uint64_t g = warp * per;
  const uint64_t g_end = min(total, g + per);
  if (g >= g_end) return;
  uint32_t lo = 0, hi = n_rec - 1; // the first record whose steps end after g
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (step_end[mid] > g) hi = mid; else lo = mid + 1;
  }
  for (uint32_t r = lo; g < g_end; r++) {
    const uint64_t r_end = step_end[r], r_begin = r ? step_end[r - 1] : 0;
    if (r_end <= g) continue;
    uint32_t len;
    const char* rec = record_of(in, r, len);
    const uint32_t c = contig_of_launch(in, r >> 1);
    const uint32_t slot = in.bf_slot ? in.bf_slot[in.contig_batch[c]] : in.contig_batch[c];
    uint32_t* const mrec = miss.bits + miss_base(in.draft_off, in.cap_off, miss.draft_words, miss.polished_words, in.nk, c, r & 1u, 0);
    const uint64_t mstride = (r & 1u) ? miss.polished_words : miss.draft_words;
    if (lane < 2 * kMaxK) acc[wib][lane >> 1][lane & 1u] = 0u;
    __syncwarp();
    uint32_t s = uint32_t(g - r_begin);
    const uint32_t s_end = uint32_t(min(g_end, r_end) - r_begin);
    uint64_t w1;
    uint32_t m1;
    pack_32(rec, len, s << 5, lane, w1, m1);
    for (; s < s_end; s++) {
      const uint64_t w0 = w1;
      const uint32_t m0 = m1;
      pack_32(rec, len, (s + 1) << 5, lane, w1, m1);
      for (uint32_t j = 0; j < in.nk; j++) {
        const StreamConsts sc = stream_consts(in.k[j]);
        const uint32_t npos = len >= sc.k ? len - sc.k + 1 : 0u;
        const uint32_t* bf = in.bf_pool + (uint64_t(slot) * in.nk + j) * kBfWords;
        bool valid = false, present = false;
        with_kmer_shape(sc, [&](auto shape) {
          uint32_t ci[4], bi[4];
          valid = hash_from_words<decltype(shape)::value>(tf, tr, w0, w1, m0, m1, s << 5, npos, lane, sc, ci, bi);
          if (valid) { // KmerBloomFilter::contains: all four bits
            const uint32_t b0 = __ldcg(bf + (bi[0] >> 5)), b1 = __ldcg(bf + (bi[1] >> 5));
            const uint32_t b2 = __ldcg(bf + (bi[2] >> 5)), b3 = __ldcg(bf + (bi[3] >> 5));
            present = ((b0 >> (bi[0] & 31u)) & (b1 >> (bi[1] & 31u)) & (b2 >> (bi[2] & 31u)) & (b3 >> (bi[3] & 31u)) & 1u) != 0u;
          }
        });
        const uint32_t vb = __ballot_sync(0xffffffffu, valid), pb = __ballot_sync(0xffffffffu, present);
        if (lane == 0) {
          acc[wib][j][0] += __popc(vb);
          acc[wib][j][1] += __popc(pb);
          mrec[j * mstride + s] = vb & ~pb;
        }
      }
    }
    __syncwarp();
    if (lane < 2 * in.nk) {
      const uint32_t j = lane >> 1, what = lane & 1u, v = acc[wib][j][what];
      if (v) atomicAdd(in.counts + (uint64_t(c) * in.nk + j) * 4 + (r & 1u) * 2 + what, (unsigned long long)v);
    }
    __syncwarp();
    g = min(g_end, r_end);
  }
}

// one block per (batch of the launch, k index): the filter's set bits
__global__ void __launch_bounds__(256) support_popcount_kernel(const uint32_t* __restrict__ bf_pool, const uint32_t* __restrict__ bf_slot,
                                                               const uint32_t* __restrict__ batches, uint32_t first_batch, uint32_t nk,
                                                               unsigned long long* __restrict__ bits)
{
  __shared__ uint32_t part[8];
  const uint32_t ib = blockIdx.x / nk, j = blockIdx.x - ib * nk;
  const uint32_t b = batches ? batches[ib] : first_batch + ib;
  const uint32_t slot = bf_slot ? bf_slot[b] : b;
  const uint4* f = reinterpret_cast<const uint4*>(bf_pool + (uint64_t(slot) * nk + j) * kBfWords);
  uint32_t n = 0;
  for (uint32_t i = threadIdx.x; i < kBfWords / 4; i += blockDim.x) {
    const uint4 v = __ldcg(f + i);
    n += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
  }
  for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31u) == 0) part[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (uint32_t w = 0; w < blockDim.x / 32; w++) t += part[w];
    bits[uint64_t(b) * nk + j] = t;
  }
}

// OR of x << d over d < k (1 <= k <= 32)
__device__ __forceinline__ uint64_t smear(uint64_t x, uint32_t k)
{
  uint32_t span = 1;
  for (; 2 * span <= k; span *= 2) x |= x << span;
  return span < k ? x | (x << (k - span)) : x;
}

// word f of the flat range: its miss bits, run starts and run lasts (covered positions followed by an uncovered one)
struct RunWord {
  uint32_t miss, starts, lasts, pos; // pos: the record position of bit 0
};

__device__ __forceinline__ RunWord run_word(const UnsupportedInput& in, uint64_t f)
{
  uint32_t lo = 0, hi = in.n_seg - 1; // the segment holding f: the last with seg_off[s] <= f
  while (lo < hi) {
    const uint32_t mid = (lo + hi + 1) >> 1;
    if (in.seg_off[mid] <= f) lo = mid; else hi = mid - 1;
  }
  const uint32_t sg = lo, j = sg % in.nk, rc = sg / in.nk, k = in.k[j];
  const uint64_t w = f - in.seg_off[sg], nw = in.seg_off[sg + 1] - in.seg_off[sg];
  const uint32_t* m = in.miss + miss_base(in.draft_off, in.cap_off, in.draft_words, in.polished_words, in.nk, rc >> 1, rc & 1u, j);
  const uint32_t cur = m[w], prev = w ? m[w - 1] : 0u, next = w + 1 < nw ? m[w + 1] : 0u;
  const uint64_t c64 = smear((uint64_t(cur) << 32) | prev, k);
  const uint32_t cov = uint32_t(c64 >> 32), cov_before = uint32_t(c64 >> 31); // bit b: position b - 1 covered
  const uint32_t next0 = uint32_t(smear((uint64_t(next) << 32) | cur, k) >> 32) & 1u;
  RunWord r;
  r.miss = cur;
  r.starts = cov & ~cov_before;
  r.lasts = cov & ~((cov >> 1) | (next0 << 31));
  r.pos = uint32_t(w) << 5;
  return r;
}

__global__ void unsupported_count_kernel(UnsupportedInput in, uint64_t n_words, uint64_t* __restrict__ run_cnt,
                                         uint32_t* __restrict__ miss_cnt)
{
  for (uint64_t f = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; f < n_words; f += uint64_t(gridDim.x) * blockDim.x) {
    const RunWord r = run_word(in, f);
    run_cnt[f] = __popc(r.starts);
    miss_cnt[f] = __popc(r.miss);
  }
}

// every start writes its run's start and subtracts the unsupported starts before it from kmers; every last writes the
// end and adds those up to and including it (both modulo 2^32: the difference is the run's count)
__global__ void unsupported_fill_kernel(UnsupportedInput in, uint64_t n_words, const uint64_t* __restrict__ run_scan,
                                        const uint32_t* __restrict__ miss_scan, gp_unsupported_run* __restrict__ runs)
{
  for (uint64_t f = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; f < n_words; f += uint64_t(gridDim.x) * blockDim.x) {
    const RunWord r = run_word(in, f);
    if (!(r.starts | r.lasts)) continue;
    const uint32_t p0 = r.pos;
    const uint64_t run0 = run_scan[f] - __popc(r.starts); // runs started before this word
    const uint32_t miss0 = miss_scan[f] - __popc(r.miss);
    for (uint32_t b = r.starts; b; b &= b - 1) {
      const uint32_t bit = __ffs(b) - 1, below = (1u << bit) - 1u;
      gp_unsupported_run& u = runs[run0 + __popc(r.starts & below)];
      u.start = p0 + bit;
      atomicAdd(&u.kmers, 0u - (miss0 + __popc(r.miss & below)));
    }
    for (uint32_t b = r.lasts; b; b &= b - 1) {
      const uint32_t bit = __ffs(b) - 1, upto = bit == 31 ? ~0u : (2u << bit) - 1u;
      gp_unsupported_run& u = runs[run0 + __popc(r.starts & upto) - 1];
      u.end = p0 + bit + 1;
      atomicAdd(&u.kmers, miss0 + __popc(r.miss & upto));
    }
  }
}

// run_off[s] = runs before segment s (s = n_seg: all of them)
__global__ void unsupported_off_kernel(const uint64_t* __restrict__ seg_off, uint32_t n_seg, const uint64_t* __restrict__ run_scan,
                                       uint64_t* __restrict__ run_off)
{
  for (uint32_t sg = blockIdx.x * blockDim.x + threadIdx.x; sg <= n_seg; sg += gridDim.x * blockDim.x)
    run_off[sg] = seg_off[sg] ? run_scan[seg_off[sg] - 1] : 0u;
}

} // namespace

// tmp == nullptr: tmp_bytes receives the scan's scratch size for in.n contigs
cudaError_t support_count(const SupportInput& in, const SupportMiss& miss, uint64_t* steps, void* tmp, size_t& tmp_bytes,
                          int sm_count, cudaStream_t s)
{
  if (!tmp) return cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, steps, steps, std::max<uint64_t>(2ull * in.n, 1), s);
  if (in.n == 0) return cudaSuccess;
  uint32_t kmin = 32;
  for (uint32_t j = 0; j < in.nk; j++) kmin = std::min(kmin, in.k[j]);
  const uint32_t n_rec = 2 * in.n;
  support_steps_kernel<<<std::min<uint32_t>((n_rec + 255) / 256, uint32_t(sm_count) * 8u), 256, 0, s>>>(in, kmin, steps);
  if (cudaError_t e = cudaGetLastError()) return e;
  if (cudaError_t e = cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, steps, steps, uint64_t(n_rec), s)) return e;
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, support_count_kernel, kSupportWarps * 32, 0);
  support_count_kernel<<<uint32_t(sm_count) * uint32_t(std::max(per_sm, 1)), kSupportWarps * 32, 0, s>>>(in, steps, miss);
  return cudaGetLastError();
}

cudaError_t support_popcount(const uint32_t* bf_pool, const uint32_t* bf_slot, const uint32_t* batches, uint32_t first_batch,
                             uint32_t n_batches, uint32_t nk, unsigned long long* bits, cudaStream_t s)
{
  if (n_batches == 0) return cudaSuccess;
  support_popcount_kernel<<<n_batches * nk, 256, 0, s>>>(bf_pool, bf_slot, batches, first_batch, nk, bits);
  return cudaGetLastError();
}

cudaError_t unsupported_count(const UnsupportedInput& in, uint64_t n_words, uint64_t* run_cnt, uint32_t* miss_cnt, void* tmp,
                              size_t& tmp_bytes, cudaStream_t s)
{
  const uint64_t n = std::max<uint64_t>(n_words, 1);
  if (!tmp) {
    size_t a = 0, b = 0;
    if (cudaError_t e = cub::DeviceScan::InclusiveSum(nullptr, a, run_cnt, run_cnt, n, s)) return e;
    if (cudaError_t e = cub::DeviceScan::InclusiveSum(nullptr, b, miss_cnt, miss_cnt, n, s)) return e;
    tmp_bytes = std::max(a, b);
    return cudaSuccess;
  }
  if (n_words == 0) return cudaSuccess;
  const uint32_t grid = uint32_t(std::min<uint64_t>((n_words + 255) / 256, 1u << 20));
  unsupported_count_kernel<<<grid, 256, 0, s>>>(in, n_words, run_cnt, miss_cnt);
  if (cudaError_t e = cudaGetLastError()) return e;
  if (cudaError_t e = cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, run_cnt, run_cnt, n_words, s)) return e;
  return cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, miss_cnt, miss_cnt, n_words, s);
}

cudaError_t unsupported_fill(const UnsupportedInput& in, uint64_t n_words, const uint64_t* run_scan, const uint32_t* miss_scan,
                             gp_unsupported_run* runs, uint64_t* run_off, cudaStream_t s)
{
  if (n_words) {
    const uint32_t grid = uint32_t(std::min<uint64_t>((n_words + 255) / 256, 1u << 20));
    unsupported_fill_kernel<<<grid, 256, 0, s>>>(in, n_words, run_scan, miss_scan, runs);
    if (cudaError_t e = cudaGetLastError()) return e;
  }
  unsupported_off_kernel<<<(in.n_seg + 256) / 256, 256, 0, s>>>(in.seg_off, in.n_seg, run_scan, run_off);
  return cudaGetLastError();
}

} // namespace gp
