// Edit records (gp_polish_fetch_edits): what the ntEdit chain changed, derived on the device from the pristine draft D,
// the polished record O and the origin map R the edit kernel composed over the k chain (R[i] = draft position of O[i],
// or GP_EDIT_INSERTED).  See include/goldpolish_b200.h for the record rules and DESIGN §4.5 for the shape.
//
// Everything is indexed by BOUNDARIES: contig c of polished length L owns L + 1 of them (boundary i sits before O[i];
// the contig's ends are virtual anchors with origins -1 and |D|), a dropped contig none.  A record starts at a boundary
// whose left side is an anchor and ends at one whose right side is an anchor; both flags come from the two positions
// around the boundary, so starts and ends pair up in order.  Pass 1 writes starts | ends << 32 per boundary and one
// exclusive scan numbers both at once; pass 2 places and normalises the records, and a scan of their allele lengths
// gives the allele offsets; pass 3 copies the allele bytes, a warp per record.
#include "gp_kernels.cuh"

#include <cub/device/device_scan.cuh>

#include <algorithm>

namespace gp {

namespace {

constexpr uint32_t kIns = GP_EDIT_INSERTED;

struct View {
  const char* D;
  const char* O;
  const uint32_t* R;
  uint32_t dlen, olen;
};

__device__ __forceinline__ View view_of(const EditsInput& in, uint32_t c)
{
  View v;
  const uint64_t d0 = in.draft_off[c];
  v.D = in.draft + d0;
  v.dlen = uint32_t(in.draft_off[c + 1] - d0);
  const uint32_t w = in.which[c];
  v.O = in.buf[w] + in.cap_off[c];
  v.R = in.orig[w] + in.cap_off[c];
  v.olen = in.len[c];
  return v;
}

__device__ __forceinline__ uint32_t up(uint32_t c) { return (c >= 'a' && c <= 'z') ? c - 32u : c; }

__device__ __forceinline__ bool is_anchor(const View& v, uint32_t i)
{
  const uint32_t r = v.R[i];
  return r != kIns && r < v.dlen && up((unsigned char)v.O[i]) == up((unsigned char)v.D[r]);
}

// the contig owning boundary g: the last c with bnd_off[c] <= g (contigs without boundaries are skipped that way)
__device__ __forceinline__ uint32_t contig_of(const uint64_t* bnd_off, uint32_t n, uint64_t g)
{
  uint32_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (bnd_off[mid] <= g) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void edits_flags_kernel(EditsInput in, uint64_t n_bnd, uint64_t* __restrict__ flags)
{
  for (uint64_t g = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; g <= n_bnd; g += uint64_t(gridDim.x) * blockDim.x) {
    if (g == n_bnd) { flags[g] = 0; continue; }
    const uint32_t c = contig_of(in.bnd_off, in.n_contigs, g);
    const View v = view_of(in, c);
    const uint32_t i = uint32_t(g - in.bnd_off[c]);
    if (i < v.olen && v.R[i] != kIns) { // origins of the non-inserted bases increase strictly and stay inside the draft
      const uint32_t r = v.R[i];
      uint32_t j = i;
      while (j > 0 && v.R[j - 1] == kIns) j--; // each run of inserted bases is walked once, by the base after it
      if (r >= v.dlen || (j > 0 && v.R[j - 1] >= r)) atomicMin(in.error, int(c) + 1);
    }
    const bool L = i == 0 || is_anchor(v, i - 1);
    const bool Rt = i == v.olen || is_anchor(v, i);
    const long long oL = i == 0 ? -1ll : (long long)v.R[i - 1];
    const long long oR = i == v.olen ? (long long)v.dlen : (long long)v.R[i];
    const bool gap = oR > oL + 1; // draft bases between the two anchors
    const uint64_t s = (L && (!Rt || gap)) ? 1u : 0u, e = (Rt && (!L || gap)) ? 1u : 0u;
    flags[g] = s | (e << 32);
  }
}

__global__ void edits_place_kernel(EditsInput in, uint64_t n_bnd, const uint64_t* __restrict__ ex, uint32_t* __restrict__ rec_c,
                                   uint32_t* __restrict__ rec_i, uint32_t* __restrict__ rec_j, uint64_t* __restrict__ contig_edit_off)
{
  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  for (uint64_t g = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; g < n_bnd; g += stride) {
    const uint64_t a = ex[g], f = ex[g + 1] - a;
    if (!f) continue;
    const uint32_t c = contig_of(in.bnd_off, in.n_contigs, g);
    const uint32_t i = uint32_t(g - in.bnd_off[c]);
    if (f & 0xFFFFFFFFull) { rec_c[uint32_t(a)] = c; rec_i[uint32_t(a)] = i; }
    if (f >> 32) rec_j[uint32_t(a >> 32)] = i;
  }
  for (uint64_t c = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; c <= in.n_contigs; c += stride)
    contig_edit_off[c] = uint32_t(ex[in.bnd_off[c]]);
}

__global__ void edits_normalise_kernel(EditsInput in, uint32_t n_rec, const uint32_t* __restrict__ rec_c,
                                       const uint32_t* __restrict__ rec_i, const uint32_t* __restrict__ rec_j,
                                       gp_edit* __restrict__ edits, uint64_t* __restrict__ alen)
{
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k <= n_rec; k += gridDim.x * blockDim.x) {
    if (k == n_rec) { alen[k] = 0; continue; }
    const View v = view_of(in, rec_c[k]);
    const uint32_t i = rec_i[k], j = rec_j[k]; // O[i, j) between the anchors O[i - 1] and O[j]
    const long long oa = i == 0 ? -1ll : (long long)v.R[i - 1];
    const long long ob = j == v.olen ? (long long)v.dlen : (long long)v.R[j];
    const uint32_t dl = uint32_t(ob - oa - 1), ol = j - i;
    gp_edit e;
    e.pos = uint32_t(oa + 1);
    e.ref_len = dl;
    e.alt_len = ol;
    if (dl && ol) e.type = dl != ol ? GP_EDIT_COMPLEX : dl == 1 ? GP_EDIT_SNV : GP_EDIT_MNV;
    else {
      e.type = dl ? GP_EDIT_DEL : GP_EDIT_INS;
      if (i > 0 || j < v.olen) { e.ref_len++; e.alt_len++; } // the left anchor's base before both, else the right one's after
      if (i > 0) e.pos = uint32_t(oa);
    }
    e.allele_off = 0;
    edits[k] = e;
    alen[k] = uint64_t(e.ref_len) + e.alt_len;
  }
}

// REF is the draft range [pos, pos + ref_len) in every case; ALT is the polished range that starts one base early when the
// left anchor was prepended (O[i - 1] equals D[pos] up to case) and runs one base on when the right one was appended
__global__ void edits_alleles_kernel(EditsInput in, uint32_t n_rec, const uint32_t* __restrict__ rec_c,
                                     const uint32_t* __restrict__ rec_i, const uint32_t* __restrict__ rec_j,
                                     const uint64_t* __restrict__ aoff, gp_edit* __restrict__ edits, char* __restrict__ alleles)
{
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_rec; k += warps) {
    const View v = view_of(in, rec_c[k]);
    const uint32_t i = rec_i[k], j = rec_j[k];
    const gp_edit e = edits[k];
    const uint32_t as = (e.alt_len > j - i && i > 0) ? i - 1 : i;
    char* dst = alleles + aoff[k];
    for (uint32_t t = lane; t < e.ref_len; t += 32) dst[t] = char(up((unsigned char)v.D[e.pos + t]));
    for (uint32_t t = lane; t < e.alt_len; t += 32) dst[e.ref_len + t] = char(up((unsigned char)v.O[as + t]));
    if (lane == 0) edits[k].allele_off = aoff[k];
  }
}

template<typename F>
uint32_t grid_for(uint64_t n, F kernel)
{
  int per_sm = 0, dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0);
  const uint64_t want = (n + 255) / 256;
  return uint32_t(std::max<uint64_t>(1, std::min<uint64_t>(want, uint64_t(std::max(sms, 1)) * std::max(per_sm, 1))));
}

} // namespace

// tmp == nullptr: tmp_bytes receives the scan's scratch size
cudaError_t edits_count(const EditsInput& in, uint64_t n_bnd, uint64_t* flags, void* tmp, size_t& tmp_bytes, cudaStream_t s)
{
  if (!tmp) return cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flags, flags, n_bnd + 1, s);
  edits_flags_kernel<<<grid_for(n_bnd + 1, edits_flags_kernel), 256, 0, s>>>(in, n_bnd, flags);
  if (cudaError_t e = cudaGetLastError()) return e;
  return cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flags, flags, n_bnd + 1, s);
}

cudaError_t edits_fill(const EditsInput& in, uint64_t n_bnd, const uint64_t* flags, uint32_t n_rec, uint32_t* rec_c,
                       uint32_t* rec_i, uint32_t* rec_j, gp_edit* edits, uint64_t* alen, uint64_t* contig_edit_off,
                       void* tmp, size_t& tmp_bytes, cudaStream_t s)
{
  if (!tmp) return cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, alen, alen, uint64_t(n_rec) + 1, s);
  edits_place_kernel<<<grid_for(std::max<uint64_t>(n_bnd, in.n_contigs + 1ull), edits_place_kernel), 256, 0, s>>>(
    in, n_bnd, flags, rec_c, rec_i, rec_j, contig_edit_off);
  if (cudaError_t e = cudaGetLastError()) return e;
  edits_normalise_kernel<<<grid_for(uint64_t(n_rec) + 1, edits_normalise_kernel), 256, 0, s>>>(in, n_rec, rec_c, rec_i, rec_j,
                                                                                                 edits, alen);
  if (cudaError_t e = cudaGetLastError()) return e;
  return cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, alen, alen, uint64_t(n_rec) + 1, s);
}

cudaError_t edits_alleles(const EditsInput& in, uint32_t n_rec, const uint32_t* rec_c, const uint32_t* rec_i,
                          const uint32_t* rec_j, const uint64_t* alen, gp_edit* edits, char* alleles, cudaStream_t s)
{
  if (n_rec == 0) return cudaSuccess;
  edits_alleles_kernel<<<grid_for(uint64_t(n_rec) * 32, edits_alleles_kernel), 256, 0, s>>>(in, n_rec, rec_c, rec_i, rec_j,
                                                                                             alen, edits, alleles);
  return cudaGetLastError();
}

} // namespace gp
