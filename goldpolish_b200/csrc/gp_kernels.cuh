// Kernel parameter blocks and launchers shared between the .cu files and the C ABI.
#pragma once

#include "../../include/goldpolish_b200.h"
#include "gp_common.cuh"

namespace gp {

constexpr int kBuildCounters = 64; // [0] k-mer ops, [1] serially resolved k-mers, [17] list entries visited, [20] / [21] first / last
                                   // globaltimer, [32..49] interval times of the level-synchronous kernel (6 kinds x {wait, work, n})
constexpr uint32_t kLevelDiag = 18, kLevelDiagAt = 32;

struct BuildParams {
  const uint64_t* pk;               // packed reads, 32 bases per word
  const uint32_t* nm;               // "no seed" mask, 32 bases per word
  const uint64_t* read_boff;        // per read: first base index (multiple of 32)
  const uint32_t* read_len;
  const uint64_t* batch_entry_off;  // global batch index -> entries
  const gp_read_entry* entries;
  uint8_t* cbf_pool;                // wave-local: stream s at s * kCbfCounters
  uint32_t* bf_pool;                // (slot * nk + ki) * kBfWords, slot = bf_slot[batch] (the batch itself without a table)
  const uint32_t* bf_slot;          // optional: pool slot of every batch (the pool is reused wave after wave)
  const uint32_t* stream_order;     // wave-local stream ids, longest first
  uint32_t* next_stream;            // work counter (zeroed before launch)
  unsigned long long* counters;     // [0] k-mer ops, [1] serially resolved k-mers
  uint32_t n_streams;
  uint32_t first_batch;
  uint32_t nk;
  uint32_t k[kMaxK];
};

constexpr uint32_t kLevelSurvWords = 3; // words per survivor-list entry: h0 low, h0 high, time | thr << 26
constexpr uint32_t kLevelListBufs = 2;  // list buffers: consecutive streams alternate

struct LevelParams {              // level-synchronous filter build (gp_build_levels.cu)
  const uint64_t* pk;
  const uint32_t* nm;
  const uint64_t* read_boff;
  const uint32_t* read_len;
  const uint64_t* batch_entry_off;
  const gp_read_entry* entries;
  const uint32_t* step_pre;       // [nk][n_entries + 1]: steps before entry e, for every k index
  const uint32_t* batch_max_thr;  // per batch: largest kmer_threshold among its entries
  const uint4* stream_tab;        // per stream of the launch, in launch order: {steps, largest thr, batch, -}
  uint32_t* batch_done;           // optional: per batch, streams whose filter is final; [n_batches_total] counts all (gp_pipeline_run)
  uint32_t n_batches_total;
  const uint16_t* anchor;         // [nk][anchor_stride]: global step of k index -> entry, relative to its batch
  uint64_t anchor_stride;
  uint32_t* V;                    // `arrays` x kCbfCounters tagged timestamps (cleared to 0xFFFFFFFF before a launch)
  uint32_t* surv;                 // kLevelListBufs x kLevelSurvWords arrays of surv_cap words, warp-private regions
  unsigned long long* bars;       // barrier arrival counter (zeroed before a launch)
  uint32_t* speed;                // per CTA: published round-0 rate (weighted shares)
  uint32_t weighted;              // 1: shares follow the measured speed of each CTA's SM
  uint32_t sms;                   // SMs of the device (set by the launch)
  uint32_t n_ctas;                // CTAs that build: keep_sms x CTAs per SM (set by the launch)
  uint32_t keep_sms;              // SMs that build: gridDim.x, or fewer (gp_pipeline_run: the others are the edit kernel's)
  uint32_t* sm_table;             // with keep_sms < sms: [0] SMs seen, [1 + 2 smid] CTAs arrived, [2 + 2 smid] rank + 1; zeroed before a launch
  uint32_t overlap;               // 1: a stream's late list rounds run beside round 0 / the level-1 round of the next stream
  uint32_t arrays;                // timestamp arrays in use: 3 (T_1 has its own: every late round can be joined), or 2 (only the last)
  uint8_t* cbf_pool;              // optional counter bytes (parity / debugging), stream s at s * kCbfCounters
  uint32_t* bf_pool;              // (slot * nk + ki) * kBfWords, slot = bf_slot[batch] (the batch itself without a table)
  const uint32_t* bf_slot;        // optional: pool slot of every batch (the pool is reused wave after wave)
  uint32_t* bf_host;              // optional: device-visible pinned host copy of ALL filters ((batch * nk + ki) * kBfWords), filled as filters become final
  unsigned long long* counters;
  unsigned long long* cta_times;  // optional: 32 words per CTA, the interval-time diagnostics of every CTA (gp_build_cta_times)
  uint32_t surv_cap;
  uint32_t time_bits;             // width of the time field of a timestamp entry (16..26): the longest stream fits
  uint32_t report_cta;            // which CTA fills the round-time diagnostics (GP_LEVEL_REPORT_CTA, default 0)
  uint32_t n_entries;
  uint32_t n_streams;
  uint32_t first_batch;
  uint32_t nk;
  uint32_t k[kMaxK];
};

struct EdNode {      // seqNode of ntedit.cpp:468-475 (num_support is never observable)
  int32_t type;      // -1 unset, 0 draft range [s, e], 1 inserted character c
  uint32_t s, e, c;
};

struct EditParams {
  uint32_t n_contigs;
  char* buf[2];                 // ping-pong sequence storage, contig i at cap_off[i]
  const uint64_t* cap_off;      // n_contigs + 1
  uint32_t* cur_len;            // in: draft length, out: polished length
  uint8_t* which;               // out: buffer index holding the result
  uint8_t* dropped;             // out: 1 if the record is not emitted
  EdNode* nodes;                // contig i at node_off[i]
  const uint64_t* node_off;     // n_contigs + 1
  const uint32_t* contig_batch;
  const uint32_t* bf_pool;      // (slot * nk + ki) * kBfWords, slot = bf_slot[batch] (the batch itself without a table)
  const uint32_t* bf_slot;
  const uint32_t* batch_done;   // optional: per batch, finished filter streams; a contig waits for nk of them ([n_batches] = total)
  uint32_t n_batches;
  const uint32_t* order;        // contig ids, longest first
  uint32_t* next_contig;
  unsigned long long* counters; // [0] triggers [1] edits [2] masked [3] rollbacks [4] first / [5] last globaltimer ns
  int* error;                   // set to 1 on buffer overflow
  uint32_t nk;
  uint32_t k[kMaxK];
  float thr_missing[kMaxK], thr_edit[kMaxK], thr_del[kMaxK];
  uint32_t insertion_cap[kMaxK];
  uint32_t max_insertions, max_deletions, jump, min_contig_len;
  int32_t mode, mask;
  uint32_t* orig[2];            // optional (gp_config.track_edits): draft position of every byte of buf[i], 4 B per byte
};                              // at 4 * cap_off[c]; orig[0] holds the identity before round 0

struct PrepParams {             // goldpolish-mask / goldpolish-to-upper on the resident contigs (gp_prep.cu)
  uint32_t n_contigs;
  char* buf[2];
  const uint64_t* cap_off;
  uint32_t* cur_len;            // in: length, out: length after masking / stripping
  uint8_t* which;               // in/out: buffer index holding the record
  const uint8_t* dropped;
  uint32_t k;                   // -k
  int32_t mode;                 // 0: to-upper only, 1: soft-mask (-s), 2: hard-mask (-n)
  int32_t to_upper;
};

void launch_pack_reads(const char* ascii, const uint64_t* ascii_off, const uint64_t* base_off, uint64_t* pk,
                       uint32_t* nm, uint32_t n_reads, cudaStream_t s);
void launch_build_filters(const BuildParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_build_filters_levels(const LevelParams& p, int sm_count, cudaStream_t s, int ctas_per_sm = 0);
int levels_ctas_per_sm(int ctas_per_sm); // CTAs the launch puts on every SM
void preload_levels();
void launch_debug_nthash(const uint64_t* pk, const uint32_t* nm, uint64_t wbase, uint32_t len, uint32_t k, uint64_t* h,
                         uint8_t* valid, cudaStream_t s);
int levels_max_grid(int sm_count, int ctas_per_sm);
void preload_edit();
void launch_fill_anchor(const uint32_t* step_pre, const uint16_t* entry_rel, uint16_t* anchor, uint32_t n_entries,
                        uint32_t nk, uint64_t anchor_stride, cudaStream_t s);
void launch_roof(uint8_t* cbf_pool, uint32_t* bf_pool, uint64_t region, uint32_t iters, uint32_t warps, cudaStream_t s);
cudaError_t launch_prep(const PrepParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_edit(const EditParams& p, int sm_count, cudaStream_t s, int alongside_build = 0); // 1: sharing SMs with the build kernel, 2: on SMs of its own

// edit records (gp_edits.cu): the polished records against the pristine draft, through the origin map
struct EditsInput {
  uint32_t n_contigs;
  const char* draft;            // pristine drafts, contig c at draft_off[c]
  const uint64_t* draft_off;    // n_contigs + 1
  const char* buf[2];           // polished record of contig c: buf[which[c]] + cap_off[c], len[c] bytes
  const uint32_t* orig[2];      // its origins: orig[which[c]] + cap_off[c]
  const uint64_t* cap_off;
  const uint32_t* len;
  const uint8_t* which;
  const uint64_t* bnd_off;      // n_contigs + 1: contig c owns the boundaries [bnd_off[c], bnd_off[c+1]) (len + 1, or 0 dropped)
  int* error;                   // out: 1 + the first contig whose origins do not increase (atomicMin; 0 = none)
};
// pass 1: flags[g] = starts | ends << 32 of boundary g (flags[G] = 0), then an exclusive scan of the G + 1 words in place
cudaError_t edits_count(const EditsInput& in, uint64_t n_bnd, uint64_t* flags, void* tmp, size_t& tmp_bytes, cudaStream_t s);
// pass 2: records into edits (pos / lengths / type) and their allele bytes into alen (n_rec + 1 words, scanned in place)
cudaError_t edits_fill(const EditsInput& in, uint64_t n_bnd, const uint64_t* flags, uint32_t n_rec, uint32_t* rec_c,
                       uint32_t* rec_i, uint32_t* rec_j, gp_edit* edits, uint64_t* alen, uint64_t* contig_edit_off,
                       void* tmp, size_t& tmp_bytes, cudaStream_t s);
// pass 3: allele bytes of every record
cudaError_t edits_alleles(const EditsInput& in, uint32_t n_rec, const uint32_t* rec_c, const uint32_t* rec_i,
                          const uint32_t* rec_j, const uint64_t* alen, gp_edit* edits, char* alleles, cudaStream_t s);

// k-mer support (gp_support.cu): the draft and the polished record of every contig of a launch against its batch's filters
struct SupportInput {
  uint32_t n;                   // contigs of this launch
  const uint32_t* ids;          // their ids (nullptr: 0 .. n - 1)
  const char* draft;            // pristine drafts, contig c at draft_off[c]
  const uint64_t* draft_off;
  const char* buf[2];           // polished record of contig c: buf[which[c]] + cap_off[c], len[c] bytes (none if dropped[c])
  const uint64_t* cap_off;
  const uint32_t* len;
  const uint8_t* which;
  const uint8_t* dropped;
  const uint32_t* contig_batch;
  const uint32_t* bf_pool;      // (slot * nk + ki) * kBfWords, slot = bf_slot[batch] (the batch itself without a table)
  const uint32_t* bf_slot;
  const int* error;             // the polish's error flag: nonzero, nothing is counted (the polish runs again)
  unsigned long long* counts;   // [contig][k index][draft k-mers, draft present, polished k-mers, polished present], added to
  uint32_t nk;
  uint32_t k[kMaxK];
};
// Unsupported k-mer starts (valid and not contained), 1 bit per start position, addressed per contig: the part of record
// r of contig c for k index j begins at word
//   r = 0 (draft):    j * draft_words + draft_off[c] / 32 + c
//   r = 1 (polished): nk * draft_words + j * polished_words + cap_off[c] / 32 + c
// with draft_words = draft_off[n] / 32 + n and polished_words = cap_off[n] / 32 + n (room for ceil(len / 32) words each)
struct SupportMiss {
  uint32_t* bits;
  uint64_t draft_words, polished_words;
};
// steps: 2 n words (record steps, scanned in place); tmp == nullptr: tmp_bytes receives the scan's scratch size.
// Every step of every record of the launch also stores its 32 unsupported-start bits per k into miss.
cudaError_t support_count(const SupportInput& in, const SupportMiss& miss, uint64_t* steps, void* tmp, size_t& tmp_bytes,
                          int sm_count, cudaStream_t s);

// Runs of unsupported k-mers (gp_polish_fetch_unsupported) from the bitmap of SupportMiss.  The words of every segment
// (contig c, record r, k index j), segment (c * 2 + r) * nk + j, form one flat range: seg_off[s] .. seg_off[s + 1]
// (ceil(len / 32) words of a record of len >= k, else none).
struct UnsupportedInput {
  const uint32_t* miss;
  uint64_t draft_words, polished_words;
  const uint64_t* draft_off;
  const uint64_t* cap_off;
  const uint64_t* seg_off;
  uint32_t n_seg;
  uint32_t nk;
  uint32_t k[kMaxK];
};
// per word of the flat range: run starts into run_cnt and unsupported starts into miss_cnt, both scanned in place
// (inclusive; miss_cnt wraps modulo 2^32, only differences inside a run are used).  tmp == nullptr: tmp_bytes receives
// the scans' scratch size.
cudaError_t unsupported_count(const UnsupportedInput& in, uint64_t n_words, uint64_t* run_cnt, uint32_t* miss_cnt, void* tmp,
                              size_t& tmp_bytes, cudaStream_t s);
// runs[] (zeroed by the caller) and run_off[0 .. n_seg] from the scanned counts
cudaError_t unsupported_fill(const UnsupportedInput& in, uint64_t n_words, const uint64_t* run_scan, const uint32_t* miss_scan,
                             gp_unsupported_run* runs, uint64_t* run_off, cudaStream_t s);
// set bits of the nk filters of n_batches batches (batches[i], or first_batch + i without a list) into bits[batch * nk + ki]
cudaError_t support_popcount(const uint32_t* bf_pool, const uint32_t* bf_slot, const uint32_t* batches, uint32_t first_batch,
                             uint32_t n_batches, uint32_t nk, unsigned long long* bits, cudaStream_t s);

} // namespace gp
