/* goldpolish_b200 -- C ABI of the B200-native GoldPolish hot path.
 *
 * Plain C, pointers and sizes only; no C++ or torch types cross this boundary.  One context
 * per GPU; calls on a context are serialised by the caller.  Every function returns 0 on
 * success or a negative gp_status; gp_last_error() gives the message.  There is no CPU
 * fallback: without a usable CUDA device gp_ctx_create fails.
 *
 * What each entry point replaces in the reference (paths relative to bcgsc/goldpolish):
 *
 *   gp_reads_upload      SeqIndex::get_seq<1> feeding fill_bfs, src/seqindex.hpp:59-102 and
 *                        src/goldpolish_targeted_bfs.cpp:130-133 (whole reads, uploaded once,
 *                        2-bit packed + validity mask on the device)
 *   gp_build_filters     serve_batch's filter loop, src/goldpolish_targeted_bfs.cpp:70-77,
 *                        124-140, i.e. fill_bfs, src/utils.cpp:96-123 (btllib::NtHash roll,
 *                        KmerCountingBloomFilter8::insert_thresh_contains, KmerBloomFilter::
 *                        insert) for every (batch, k); bf_out payloads are what
 *                        KmerBloomFilter::save writes after its text header (:138-140)
 *   gp_filters_load      btllib::KmerBloomFilter(path) payload, subprojects/ntedit/
 *                        ntedit.cpp:2012-2022 (lets ntedit-gr run on filters built elsewhere)
 *   gp_polish            readAndCorrect + kmerizeAndCorrect + writeEditsToFile for every
 *                        contig, subprojects/ntedit/ntedit.cpp:1414-1867, chained over the
 *                        context's k list as scripts/goldpolish-ntedit:20-29 chains processes
 *   gp_guard_rejects     the 0.75 size guard, scripts/goldpolish-ntedit:31-40
 *   gp_flagged_bed       the soft-masked ("flagged") regions of ntEdit -a1, subprojects/ntedit/ntedit.cpp:1131-1146,
 *                        as BED intervals (the reference itself only lower-cases the bases)
 *   gp_polish_fetch_edits  what polishing changed, per contig, in draft coordinates (VCF-normalised records).  The
 *                        reference fork writes no such file: its writeEditsToFile pops the substitution records and
 *                        writes the FASTA only (subprojects/ntedit/ntedit.cpp:797-935; upstream ntEdit's _changes.tsv
 *                        is gone).  DERIVED from the polished record and a map of each polished base to its draft
 *                        position, composed over the k chain as the edit kernel copies the bases
 *   gp_kmer_threshold    mappings_bases_to_kmer_threshold, src/goldpolish_targeted_bfs.cpp:45-53
 *   gp_mappings_cap      mappings_num_max, src/goldpolish_targeted_bfs.cpp:96-99
 */
#ifndef GOLDPOLISH_B200_H
#define GOLDPOLISH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GP_MAX_K_VALUES 8
#define GP_CBF_BYTES 10485760ULL /* src/goldpolish_targeted_bfs.cpp:270 */
#define GP_BF_BYTES 524288ULL    /* src/goldpolish_targeted_bfs.cpp:271 */
#define GP_HASH_NUM 4u           /* src/goldpolish_targeted_bfs.cpp:272 */

typedef enum {
  GP_OK = 0,
  GP_ERR_ARG = -1,      /* bad argument / unsupported configuration */
  GP_ERR_CUDA = -2,     /* CUDA runtime error (message holds cudaGetErrorString) */
  GP_ERR_NO_DEVICE = -3,/* no CUDA device: this library has no CPU path */
  GP_ERR_OOM = -4,      /* device or host allocation failed */
  GP_ERR_STATE = -5,    /* call order (e.g. polish before filters exist) */
  GP_ERR_OVERFLOW = -6  /* an edited contig outgrew its device buffers */
} gp_status;

typedef struct gp_ctx gp_ctx;

typedef struct {
  uint32_t struct_size;            /* sizeof(gp_config), for ABI growth */
  int32_t device;                  /* CUDA device ordinal */
  uint32_t nk;                     /* number of k values (<= GP_MAX_K_VALUES) */
  uint32_t k[GP_MAX_K_VALUES];     /* descending, e.g. 32 28 24 20; each 4..32 */
  /* ntEdit options, defaults = scripts/goldpolish-ntedit:27 (-d5 -i5 -m1 -X0.5 -Y0.5 -a1) */
  uint32_t max_insertions;         /* -i, 0..5 */
  uint32_t max_deletions;          /* -d, 0..10 */
  int32_t mode;                    /* -m, 0..2 */
  int32_t mask;                    /* -a */
  float missing_ratio;             /* -X */
  float edit_ratio;                /* -Y */
  uint32_t jump;                   /* -j */
  uint32_t min_contig_len;         /* -z */
  uint32_t max_resident_batches;   /* cap on batches whose counting filters live at once; 0 = fit to free memory */
  int32_t use_ratio;               /* 1: thresholds from -X/-Y (default); 0: from -x/-y below */
  float missing_threshold;         /* -x */
  float edit_threshold;            /* -y */
  int32_t keep_counters;           /* 1: also materialise the counting-filter bytes (gp_build_fetch_cbf; parity tests) */
  /* optional post-pass on the polished records while they are still on the device (default off):
   * goldpolish-mask (scripts/goldpolish-mask:44-72) and goldpolish-to-upper (scripts/goldpolish-to-upper:15-21) */
  int32_t prep_mode;               /* 0 off, 1 = goldpolish-mask -s (soft), 2 = goldpolish-mask -n (hard) */
  uint32_t prep_k;                 /* its -k (scripts/goldpolish-make:66 passes the first k value); 1..64 */
  int32_t to_upper;                /* 1: upper-case the records (after masking, if any) */
  /* cap on batches whose Bloom filters (nk x 512 KiB each) are resident at once; 0 = every batch of a call when they fit
   * (at most half of the free device memory), else as many as fit.  When fewer than all are resident the pool is reused
   * wave after wave: gp_pipeline_run polishes every wave before its filters go and gp_build_output_host receives the
   * payloads; gp_build_run needs that destination, and a separate gp_polish is not possible. */
  uint32_t max_resident_filters;
  /* 1: follow every polished base back to the draft position it came from, so that gp_polish_fetch_edits can report
   * the edits (default 0).  Not combinable with prep_mode 2: hard-masked bases would read as substitutions. */
  int32_t track_edits;
} gp_config;

/* one read handed to fill_bfs: index into the uploaded read store + the target's kmer_threshold */
typedef struct {
  uint32_t read_id;
  uint32_t kmer_threshold; /* T of goldpolish_targeted_bfs.cpp:124-125; fill_bfs uses T-2+idx(k) */
} gp_read_entry;

typedef struct {
  uint64_t kmer_ops;        /* valid (read k-mer, k) pairs processed by the last build */
  uint64_t serial_kmers;    /* of those, resolved on the in-order (colliding) path */
  uint64_t triggers;        /* ntEdit: absent k-mers that started an edit attempt (last polish) */
  uint64_t edits;           /* substitutions + insertions + deletions applied */
  uint64_t masked;          /* soft-masked positions */
  uint64_t rollbacks;       /* low-complexity insertion rollbacks */
  float build_ms;           /* device time of the last build (CUDA events on the ctx stream) */
  float polish_ms;          /* device time of the last polish */
  float pack_ms;            /* device time of the last read packing */
  float build_kernel_ms;    /* of build_ms, the filter-build kernel alone (memsets excluded) */
  float edit_kernel_ms;     /* of polish_ms, the edit kernel alone */
  uint32_t build_launches;  /* kernels (not memsets) launched by the last build */
  uint32_t polish_launches; /* kernels launched by the last polish */
  uint32_t pack_launches;
  uint32_t build_kernel;    /* which filter-build kernel ran: 1 = one warp per stream (in order, counters in HBM),
                               2 = level-synchronous (order-free rounds, timestamps in L2) */
  uint32_t build_slots;     /* level-synchronous kernel: streams in flight */
  uint32_t polish_reruns;   /* times gp_polish_fetch had to run the polish again since the context was created
                               (a contig outgrew its buffers, or the overlapped edit kernel's watchdog fired) */
  uint32_t edit_sms;        /* last gp_pipeline_run: SMs the edit kernel had to itself beside the build kernel
                               (0: the two kernels shared every SM, or nothing was overlapped) */
  uint32_t level_time_bits; /* last build: width of the occurrence times of the level-synchronous kernel (the epoch tags
                               take the other 32 - level_time_bits bits); 0 when the in-order kernel ran */
} gp_stats;

void gp_default_config(gp_config* cfg);
int gp_ctx_create(const gp_config* cfg, gp_ctx** out);
void gp_ctx_destroy(gp_ctx* ctx);
const char* gp_last_error(const gp_ctx* ctx); /* ctx may be NULL: error of the last failed create */

/* Run all work of this context on an existing CUDA stream (a cudaStream_t passed as void*),
 * e.g. so that a caller's CUDA events bracket it.  NULL restores the context's own stream. */
int gp_ctx_set_stream(gp_ctx* ctx, void* cuda_stream);
int gp_ctx_synchronize(gp_ctx* ctx);
int gp_get_stats(const gp_ctx* ctx, gp_stats* out);

/* ---- read store ------------------------------------------------------------------- */
/* seqs: ASCII bases of all reads back to back; read i = seqs[offsets[i] .. offsets[i+1]).
 * Host buffers; copied to the device and packed there.  Replaces any previous store. */
int gp_reads_upload(gp_ctx* ctx, const char* seqs, const uint64_t* offsets, uint64_t n_reads);
/* The same store filled piecewise, for callers that read sequences from a file as they go (the reference reads every
 * sequence on demand, src/seqindex.hpp:59-102): announce all read lengths, then append the bases of consecutive reads
 * (back to back, any number of reads per call, in read order), then end.  Neither side ever holds the whole read set
 * as text: the device stages at most 256 MiB (or the longest read) of ASCII per slab, packs it (2 bits + 1 mask bit per
 * base) and reuses the staging; gp_reads_upload is begin + one append + end.  Replaces any previous store. */
int gp_reads_begin(gp_ctx* ctx, uint64_t n_reads, const uint32_t* lens);
int gp_reads_append(gp_ctx* ctx, const char* seqs, uint64_t n_reads_in_this_call);
int gp_reads_end(gp_ctx* ctx);

/* ---- filter build ----------------------------------------------------------------- */
/* Batch b hashes entries[batch_entry_off[b] .. batch_entry_off[b+1]) in that order, every read
 * with every k of the context, into its own nk (counting filter, filter) pairs.
 * bf_out (host, may be NULL): n_batches * nk * GP_BF_BYTES payload bytes, batch-major then k.
 * The filters stay resident as the context's current filter set for gp_polish. */
int gp_build_filters(gp_ctx* ctx, uint32_t n_batches, const uint64_t* batch_entry_off,
                     const gp_read_entry* entries, uint8_t* bf_out);

/* split form of the same call (stage = host->device copies, run = kernels only,
 * fetch = device->host copy); gp_build_filters == stage + run + fetch */
int gp_build_stage(gp_ctx* ctx, uint32_t n_batches, const uint64_t* batch_entry_off, const gp_read_entry* entries);
int gp_build_run(gp_ctx* ctx);
/* Optional: name a PAGE-LOCKED host buffer (n_batches * nk * GP_BF_BYTES of the builds to come) as the destination
 * of the filter payloads.  The level-synchronous build kernel then writes every filter there itself the moment it
 * is final (each CTA stores its slice over PCIe under the following rounds), and gp_build_fetch(ctx, same pointer)
 * only synchronises -- no bulk D2H after the build.  NULL switches it off.  What the reference does per batch with
 * bfs[i]->save() (goldpolish_targeted_bfs.cpp:138-140), without the end-of-build wait. */
int gp_build_output_host(gp_ctx* ctx, uint8_t* bf_out_pinned);
/* Page-locked host memory for callers that do not link the CUDA runtime themselves (the C++ drop-in tools):
 * NULL when it cannot be had.  A context must exist (the device is chosen by then). */
void* gp_host_alloc(uint64_t bytes);
void gp_host_free(void* p);
int gp_build_fetch(gp_ctx* ctx, uint8_t* bf_out);
/* debug / parity: counting-filter bytes of (batch, k index) after the last build */
int gp_build_fetch_cbf(gp_ctx* ctx, uint32_t batch, uint32_t k_index, uint8_t* cbf_out);

/* Make externally built payloads (n_batches * nk * GP_BF_BYTES) the current filter set. */
int gp_filters_load(gp_ctx* ctx, uint32_t n_batches, const uint8_t* bf_payloads);

/* ---- polish ----------------------------------------------------------------------- */
/* Contig i = seqs[offsets[i] .. offsets[i+1]) uses the filters of batch contig_batch[i] and is
 * run through every k of the context in order.  Outputs (host): out_seqs/out_offsets in CSR
 * form (a dropped contig has an empty range), out_dropped[i] = 1 when the reference would not
 * emit the record (shorter than min_contig_len at any round, ntedit.cpp:1850).
 * Returns GP_ERR_ARG if out_cap is too small (needed size in out_offsets[n_contigs]). */
int gp_polish(gp_ctx* ctx, uint32_t n_contigs, const char* seqs, const uint64_t* offsets,
              const uint32_t* contig_batch, char* out_seqs, uint64_t out_cap, uint64_t* out_offsets,
              uint8_t* out_dropped);

int gp_polish_stage(gp_ctx* ctx, uint32_t n_contigs, const char* seqs, const uint64_t* offsets,
                    const uint32_t* contig_batch);
int gp_polish_run(gp_ctx* ctx);
int gp_polish_fetch(gp_ctx* ctx, char* out_seqs, uint64_t out_cap, uint64_t* out_offsets, uint8_t* out_dropped);

/* goldpolish-mask / goldpolish-to-upper alone (no filters needed): records in, records out.  mode and k as
 * gp_config.prep_mode / prep_k (mode 0 = to-upper only); out_offsets has n_records + 1 entries. */
int gp_prep(gp_ctx* ctx, uint32_t n_records, const char* seqs, const uint64_t* offsets, int32_t mode, uint32_t k,
            int32_t to_upper, char* out_seqs, uint64_t out_cap, uint64_t* out_offsets);

/* gp_build_run + gp_polish_run of the staged work as ONE overlapped pass (needs gp_build_stage and
 * gp_polish_stage first; results are fetched with gp_build_fetch / gp_polish_fetch as usual and are
 * identical to the two separate calls).  The batches holding the longest contigs are built first, and a
 * persistent edit kernel -- launched behind the build kernel in the same stream with programmatic stream
 * serialization, so that it becomes resident beside it -- starts on each contig as soon as the nk filters of
 * its batch are final: the reference's per-batch order "BF server answers, then goldpolish-ntedit runs"
 * (scripts/goldpolish-polish-batch:62-105), kept per batch instead of per run.  The edit kernel runs on a few SMs of
 * its own, which the build launch hands back (gp_stats.edit_sms; environment GP_EDIT_SMS=n fixes their number, 0 makes
 * the two kernels share every SM).  Falls back to the two calls in sequence when there is nothing to overlap (in-order
 * build kernel, keep_counters) or when the device turned out not to co-schedule the two kernels (the edit kernel's
 * watchdog, checked after the first pass). */
int gp_pipeline_run(gp_ctx* ctx);

/* ---- edit records ------------------------------------------------------------------- */
/* With cfg.track_edits the edit kernel maps every polished base to its 0-based position in the ORIGINAL draft contig, or
 * to GP_EDIT_INSERTED, composing the map over the k chain.  An anchor is a polished base that maps to a draft base
 * equal to it up to case (soft-masking is not an edit).  Each gap between consecutive anchors (the contig's ends count
 * as anchors) whose draft span D or polished span O is non-empty is ONE record, normalised as VCF does:
 *   D and O non-empty: pos = first base of D, ref = D, alt = O (SNV 1/1, MNV n/n, COMPLEX otherwise);
 *   one of them empty: the left anchor's draft base is prepended to both and pos is that base (INS / DEL); at the
 *   contig start the right anchor's base is appended instead.
 * ref and alt are upper-cased.  Changes that cancel over the chain (a base inserted at one k, deleted at the next)
 * leave no record: the records say what the polished record changed against the draft.  The records describe the
 * ntEdit chain's output, before the optional goldpolish-mask / to-upper post-pass.  Origins that do not increase along
 * a contig are an internal error (GP_ERR_STATE), never a silently wrong record. */
#define GP_EDIT_INSERTED 0xFFFFFFFFu
#define GP_EDIT_SNV 0u
#define GP_EDIT_MNV 1u
#define GP_EDIT_INS 2u
#define GP_EDIT_DEL 3u
#define GP_EDIT_COMPLEX 4u
typedef struct { uint32_t pos, ref_len, alt_len, type; uint64_t allele_off; } gp_edit; /* REF then ALT bytes at alleles[allele_off] */
/* records of the last gp_polish / gp_pipeline_run, contig order then pos; needs cfg.track_edits.  Like gp_polish_fetch
 * they come before the 0.75 guard, and a dropped contig has none.
 * contig_edit_off: n_contigs + 1 (CSR).  Too-small caps -> GP_ERR_ARG with needed[0] = records, needed[1] = allele bytes
 * (contig_edit_off is filled either way; edits / alleles may be NULL with a cap of 0). */
int gp_polish_fetch_edits(gp_ctx* ctx, uint64_t* contig_edit_off, gp_edit* edits, uint64_t edits_cap,
                          char* alleles, uint64_t alleles_cap, uint64_t needed[2]);

/* ---- flagged regions ---------------------------------------------------------------- */
/* The reference flags what it could not fix by soft-masking: ntEdit -a1 lower-cases the draft base at every position
 * whose k-mer stayed absent (subprojects/ntedit/ntedit.cpp:1131-1146; the flag is passed at scripts/goldpolish-ntedit:27)
 * and writes NO BED file of its own.  The flagged-region BED is therefore DERIVED from the polished FASTA: one
 * interval per maximal run of lower-case letters, 0-based half-open [start, end) in the coordinates of the polished
 * record.  (Lower-case bases that were already soft-masked in the input survive polishing and are reported too.)
 * Pure host code: records in CSR form as gp_polish returns them; fills record index / start / end of up to `cap`
 * runs in record order and returns the total number of runs (call again with a larger cap if it exceeds cap). */
uint64_t gp_flagged_bed(const char* seqs, const uint64_t* offsets, uint32_t n_records, uint32_t* run_record,
                        uint64_t* run_start, uint64_t* run_end, uint64_t cap);

/* ---- host-side rules shared with the reference ------------------------------------ */
int gp_kmer_threshold(uint64_t mappings_bases);
uint64_t gp_mappings_cap(uint64_t target_len, double subsample_max_per_10kbp);
int gp_guard_rejects(uint64_t input_bytes, uint64_t output_bytes);

/* ---- measurement support ---------------------------------------------------------- */
/* Random-access roof microbenchmark with the build kernel's access shape: `warps` warps, each
 * doing `iters` rounds of 32x4 dependent byte loads + conditional byte stores into a private
 * region of region_bytes, plus 32x4 atomicOr into a private 512 KiB region.  Returns sector
 * touches per second (8 per k-mer op) in *sectors_per_s.  Environment GP_ROOF_MODE selects other shapes:
 * 1 loads only, 2 loads + counter stores (HBM, private regions); 3 alternating rounds of 4 atomicMin / 4 loads,
 * 4 atomicMin only, 5 loads only over ONE shared 40 MiB array in L2 (the level-synchronous kernel's shape;
 * 4 touches per iteration are counted). */
int gp_roof_microbench(gp_ctx* ctx, uint32_t warps, uint32_t iters, uint64_t region_bytes, double* sectors_per_s,
                       float* ms);

/* Known-answer support: the four ntHash values (btllib::NtHash::hashes(), spec in subprojects/ntedit/lib/nthash.hpp:
 * 293-314) of every k-mer start of uploaded read `read_id`, computed by the device code the build kernels use (2-bit
 * packed words + mask window, shared-memory byte tables, multiply-xorshift extra hashes).  hashes[4 p .. 4 p + 3] and
 * valid[p] (0: the k-mer holds a non-ACGT base and is skipped, as NtHash::roll does) for p < *n_positions = len-k+1. */
int gp_debug_nthash(gp_ctx* ctx, uint64_t read_id, uint32_t k, uint64_t* hashes, uint8_t* valid, uint64_t cap_positions,
                    uint64_t* n_positions);

/* Diagnostic (no reference counterpart): where the time of one CTA of the level-synchronous build
 * kernel went during the last gp_build_run, per kind of barrier interval r = 0 clear, 1 round 0 alone (hashing +
 * first timestamps), 2 the level-1 list round alone, 3 a late list round alone, 4 round 0 beside the previous
 * stream's last round, 5 the level-1 round beside it: out[3r] = ns waiting at the grid barrier, out[3r+1] = ns working,
 * out[3r+2] = intervals; out[31] = survivor-list entries visited by all list rounds. */
int gp_build_round_times(gp_ctx* ctx, uint64_t out[32]);
/* The same numbers for EVERY CTA of the last level-synchronous launch (32 words per CTA, laid out as above),
 * recorded only when the environment variable GP_LEVEL_CTA_TIMES is set: shows which CTAs the grid barrier waits for. */
int gp_build_cta_times(gp_ctx* ctx, uint64_t* out, uint32_t cap_ctas, uint32_t* n_ctas);

#ifdef __cplusplus
}
#endif
#endif
