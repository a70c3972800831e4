// C ABI of goldpolish_b200 (see include/goldpolish_b200.h for the reference mapping).
// Host-side plumbing only: device buffers, staging copies, wave scheduling, kernel launches.
#include "gp_kernels.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

namespace {

thread_local std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t need)
  {
    if (need <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = need + need / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { cudaGetLastError(); e = cudaMalloc(&p, need); want = need; }
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template<typename T> T* as() const { return static_cast<T*>(p); }
};

} // namespace

struct gp_ctx {
  gp_config cfg;
  int sm_count = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  uint8_t* bf_host_user = nullptr;                    // gp_build_output_host: pinned destination of the filter payloads
  uint32_t* bf_host_dev = nullptr;                    // ... as the device sees it
  bool bf_streamed = false;                           // the last build wrote the payloads there itself
  std::vector<uint32_t> h_pre, h_maxthr;              // steps before every entry per k; largest kmer_threshold per batch
  std::vector<uint64_t> h_batch_entry_off;
  std::vector<uint4> h_stream_tab;
  DevBuf d_stream_tab;
  std::vector<uint32_t> h_empty_streams;              // (batch * nk + ki) of streams without a k-mer
  bool edit_ev_valid = false;                         // edit_ev[] were recorded by the last polish
  int l2_persist_max = 0, l2_window_max = 0;          // persisting-L2 capacity and largest access-policy window (bytes)
  bool l2_window_set = false, l2_roof_window = false;
  int overlap_state = 0;                              // 0 untested, 1 the two kernels co-run on this device, -1 they do not
  bool pipelined = false;                             // last run was gp_pipeline_run's overlapped pass (device timers)
  cudaEvent_t ev[6] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr }; // pack, build, polish (start, stop)
  std::vector<cudaEvent_t> wave_ev;  // build kernel only: (start, stop) per wave
  cudaEvent_t edit_ev[2] = { nullptr, nullptr }; // edit kernel only
  std::string err;
  gp_stats stats;
  bool build_timed = false, polish_timed = false, pack_timed = false;

  // read store
  uint64_t n_reads = 0;
  uint64_t reads_total = 0, reads_next = 0, read_slab = 0; // gp_reads_begin / _append / _end in progress
  std::vector<uint32_t> h_read_len;
  std::vector<uint64_t> h_read_boff;
  DevBuf d_ascii, d_ascii_off, d_pk, d_nm, d_read_boff, d_read_len;

  // build
  uint32_t n_batches = 0;      // batches of the current filter set
  bool filters_ready = false; // the context's current filter set is resident (gp_polish can run)
  bool build_done = false;    // a staged build has run (its payloads can be fetched)
  bool build_staged = false;
  uint32_t wave_batches = 0;
  bool bf_all_resident = true;                        // the filter pool holds every batch of the call (else: one wave at a time)
  std::vector<uint32_t> h_bf_slot;                    // pool slot of every batch when it does not
  DevBuf d_bf_slot;
  std::vector<uint32_t> wave_first, wave_count, wave_order_off;
  DevBuf d_batch_entry_off, d_entries, d_bf_pool, d_cbf_pool, d_stream_order, d_next, d_counters;
  // level-synchronous build
  DevBuf d_step_pre, d_batch_max_thr, d_V, d_alive, d_anchor, d_entry_rel, d_cta_times, d_sm_table;
  uint32_t edit_sms = 0;   // SMs that the last overlapped pass gave to the edit kernel (0: the two kernels shared every SM)
  uint32_t edit_ctas_per_sm = 0; // build CTAs per SM of that pass
  int sm_split_state = 0;  // 0 unchecked, 1 the build launch vacates whole SMs on this device (checked), -1 it does not
  uint32_t level_grid = 0; // CTAs of the last level-synchronous launch
  uint64_t anchor_stride = 0;
  uint32_t alive_words = 0, n_entries = 0, surv_cap = 0, level_slots = 1, level_time_bits = 26, level_arrays = 2;
  bool levels_ok = false; // every stream fits the 26-bit occurrence clock
  int build_algo = 0;     // 0 = auto, 1 = warp per stream, 2 = level-synchronous
  int build_algo_resolved = 1;

  // polish
  uint32_t n_contigs = 0;
  bool polish_staged = false, polish_done = false;
  uint32_t grow = 0; // overflow retries enlarge the buffers
  std::vector<uint64_t> h_in_off, h_cap_off, h_node_off;
  std::vector<uint32_t> h_len, h_order, h_batch;
  std::vector<uint32_t> h_batch_order, h_order_pipe;  // gp_pipeline_run: batches / contigs in build order
  std::vector<uint32_t> h_wave_contig_off;            // ... and where every wave's contigs start in h_order_pipe
  DevBuf d_batch_order, d_batch_done, d_order_pipe;
  DevBuf d_input, d_in_off, d_buf0, d_buf1, d_cap_off, d_cur_len, d_which, d_dropped, d_nodes, d_node_off,
    d_contig_batch, d_order, d_pnext, d_pcounters, d_error, d_out, d_out_off;

  // edit records (cfg.track_edits): origin slices beside d_buf0 / d_buf1, the edit kernel's own result (the optional
  // mask / to-upper pass moves the records on), and the records derived from them, kept until the next polish
  bool edits_polish = false;  // the last polish ran with tracking (its records can be derived)
  bool edits_ready = false;   // ... and they have been
  uint64_t n_edits = 0, n_allele_bytes = 0;
  DevBuf d_orig0, d_orig1, d_elen, d_ewhich, d_bnd_off, d_eflags, d_etmp, d_rec_c, d_rec_i, d_rec_j, d_edits, d_alen,
    d_alleles, d_edit_coff, d_edit_err;

  // k-mer support (cfg.kmer_support): per (contig, k) counts and per (batch, k) set bits, taken in stream order after the
  // edit kernel of every launch (every wave) while its filters are resident, before the mask / to-upper pass
  bool support_polish = false; // the last polish counted them
  DevBuf d_support, d_sup_steps, d_sup_tmp, d_sup_bits;
  // where the unsupported k-mers lie: the count kernel's bitmap (gp::SupportMiss) and the polished lengths it saw; the
  // runs derived from them at the first gp_polish_fetch_unsupported
  uint64_t sup_draft_words = 0, sup_polished_words = 0;
  bool unsupported_ready = false;
  uint64_t n_unsupported = 0;
  DevBuf d_sup_miss, d_sup_len, d_uns_seg, d_uns_runcnt, d_uns_misscnt, d_uns_tmp, d_uns_runs, d_uns_off;
};

#define GP_FAIL(ctx, code, msg)                                                                              \
  do {                                                                                                       \
    (ctx)->err = (msg);                                                                                      \
    return (code);                                                                                           \
  } while (0)

#define GP_CUDA(ctx, call)                                                                                   \
  do {                                                                                                       \
    cudaError_t e_ = (call);                                                                                 \
    if (e_ != cudaSuccess) {                                                                                 \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                       \
      cudaGetLastError();                                                                                    \
      return e_ == cudaErrorMemoryAllocation ? GP_ERR_OOM : GP_ERR_CUDA;                                     \
    }                                                                                                        \
  } while (0)

namespace {

// small device helpers that do not belong to a hot kernel -------------------------------
__global__ void scatter_contigs_kernel(const char* __restrict__ in, const uint64_t* __restrict__ in_off,
                                       char* __restrict__ buf0, const uint64_t* __restrict__ cap_off,
                                       uint32_t* __restrict__ cur_len, uint32_t* __restrict__ orig0, uint32_t n)
{
  for (uint32_t c = blockIdx.x; c < n; c += gridDim.x) {
    const uint64_t a = in_off[c];
    const uint32_t len = uint32_t(in_off[c + 1] - a);
    char* dst = buf0 + cap_off[c];
    for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) dst[i] = in[a + i];
    if (orig0) // edit records: round 0 starts from the identity
      for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) orig0[cap_off[c] + i] = i;
    if (threadIdx.x == 0) cur_len[c] = len;
  }
}

__global__ void gather_contigs_kernel(const char* __restrict__ buf0, const char* __restrict__ buf1,
                                      const uint64_t* __restrict__ cap_off, const uint8_t* __restrict__ which,
                                      const uint64_t* __restrict__ out_off, char* __restrict__ out, uint32_t n)
{
  for (uint32_t c = blockIdx.x; c < n; c += gridDim.x) {
    const uint64_t o = out_off[c];
    const uint32_t len = uint32_t(out_off[c + 1] - o);
    const char* src = (which[c] ? buf1 : buf0) + cap_off[c];
    for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) out[o + i] = src[i];
  }
}

int validate_config(const gp_config& c, std::string& why)
{
  if (c.nk == 0 || c.nk > GP_MAX_K_VALUES) { why = "nk must be 1..8"; return GP_ERR_ARG; }
  for (uint32_t i = 0; i < c.nk; i++)
    if (c.k[i] < 4 || c.k[i] > 32) { why = "k must be within 4..32"; return GP_ERR_ARG; }
  if (c.max_insertions > 5) { why = "max_insertions must be <= 5"; return GP_ERR_ARG; }
  if (c.max_deletions > 10) { why = "max_deletions must be <= 10"; return GP_ERR_ARG; }
  if (c.mode < 0 || c.mode > 2) { why = "mode must be 0..2"; return GP_ERR_ARG; }
  if (c.jump == 0) { why = "jump must be >= 1"; return GP_ERR_ARG; }
  if (c.prep_mode < 0 || c.prep_mode > 2) { why = "prep_mode must be 0..2"; return GP_ERR_ARG; }
  if (c.prep_mode && (c.prep_k == 0 || c.prep_k > 64)) { why = "prep_k must be within 1..64"; return GP_ERR_ARG; }
  if (!c.use_ratio && (!(c.missing_threshold > 0) || !(c.edit_threshold > 0))) { why = "x / y thresholds must be > 0"; return GP_ERR_ARG; }
  if (c.kmer_support < 0 || c.kmer_support > 1) { why = "kmer_support must be 0 or 1"; return GP_ERR_ARG; }
  if (c.track_edits && c.prep_mode == 2) { why = "track_edits cannot be combined with prep_mode 2 (hard-masked bases would read as substitutions)"; return GP_ERR_ARG; }
  return GP_OK;
}

} // namespace

extern "C" {

void gp_default_config(gp_config* cfg)
{
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->struct_size = sizeof(gp_config);
  cfg->device = 0;
  cfg->nk = 4;
  cfg->k[0] = 32; cfg->k[1] = 28; cfg->k[2] = 24; cfg->k[3] = 20; // scripts/goldpolish:189-190
  cfg->max_insertions = 5; cfg->max_deletions = 5; cfg->mode = 1; cfg->mask = 1; // scripts/goldpolish-ntedit:27
  cfg->missing_ratio = 0.5f; cfg->edit_ratio = 0.5f;
  cfg->use_ratio = 1;                                        // GoldPolish always passes -X/-Y
  cfg->missing_threshold = 5.0f; cfg->edit_threshold = 9.0f; // ntedit.cpp:88-89
  cfg->jump = 3; cfg->min_contig_len = 100; // ntedit.cpp:94,85
  cfg->max_resident_batches = 0;
  cfg->track_edits = 0; cfg->kmer_support = 0; // extensions without a reference counterpart: off
}

const char* gp_last_error(const gp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int gp_ctx_create(const gp_config* cfg, gp_ctx** out)
{
  if (!cfg || !out) { g_create_error = "null argument"; return GP_ERR_ARG; }
  *out = nullptr;
  gp_config c;
  gp_default_config(&c);
  std::memcpy(&c, cfg, std::min<size_t>(cfg->struct_size ? cfg->struct_size : sizeof(gp_config), sizeof(gp_config)));
  c.struct_size = sizeof(gp_config);
  std::string why;
  if (int rc = validate_config(c, why)) { g_create_error = why; return rc; }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) +
                     "); goldpolish_b200 has no CPU path";
    return GP_ERR_NO_DEVICE;
  }
  if (c.device < 0 || c.device >= ndev) { g_create_error = "device ordinal out of range"; return GP_ERR_ARG; }
  if ((e = cudaSetDevice(c.device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return GP_ERR_CUDA; }
  gp_ctx* ctx = new gp_ctx();
  ctx->cfg = c;
  std::memset(&ctx->stats, 0, sizeof(ctx->stats));
  cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, c.device);
  cudaDeviceGetAttribute(&ctx->l2_persist_max, cudaDevAttrMaxPersistingL2CacheSize, c.device);
  cudaDeviceGetAttribute(&ctx->l2_window_max, cudaDevAttrMaxAccessPolicyWindowSize, c.device);

  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_create_error = cudaGetErrorString(e);
    delete ctx;
    return GP_ERR_CUDA;
  }
  ctx->stream = ctx->own_stream;
  gp::preload_levels(); // (CUDA loads kernels lazily; the first overlapped pass must not stall on that)
  gp::preload_edit();
  for (auto& ev : ctx->ev) cudaEventCreate(&ev);
  for (auto& ev : ctx->edit_ev) cudaEventCreate(&ev);
  *out = ctx;
  return GP_OK;
}

void gp_ctx_destroy(gp_ctx* ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->cfg.device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf* bufs[] = { &ctx->d_ascii, &ctx->d_ascii_off, &ctx->d_pk, &ctx->d_nm, &ctx->d_read_boff, &ctx->d_read_len,
                     &ctx->d_batch_entry_off, &ctx->d_entries, &ctx->d_bf_pool, &ctx->d_cbf_pool, &ctx->d_stream_order,
                     &ctx->d_next, &ctx->d_counters, &ctx->d_step_pre, &ctx->d_batch_max_thr, &ctx->d_V, &ctx->d_alive, &ctx->d_anchor, &ctx->d_entry_rel, &ctx->d_input, &ctx->d_in_off, &ctx->d_buf0, &ctx->d_buf1,
                     &ctx->d_cap_off, &ctx->d_cur_len, &ctx->d_which, &ctx->d_dropped, &ctx->d_nodes, &ctx->d_node_off,
                     &ctx->d_contig_batch, &ctx->d_order, &ctx->d_pnext, &ctx->d_pcounters, &ctx->d_error, &ctx->d_out,
                     &ctx->d_out_off, &ctx->d_batch_order, &ctx->d_batch_done, &ctx->d_order_pipe, &ctx->d_stream_tab, &ctx->d_cta_times, &ctx->d_bf_slot,
                     &ctx->d_orig0, &ctx->d_orig1, &ctx->d_elen, &ctx->d_ewhich, &ctx->d_bnd_off, &ctx->d_eflags, &ctx->d_etmp,
                     &ctx->d_rec_c, &ctx->d_rec_i, &ctx->d_rec_j, &ctx->d_edits, &ctx->d_alen, &ctx->d_alleles, &ctx->d_edit_coff,
                     &ctx->d_edit_err, &ctx->d_support, &ctx->d_sup_steps, &ctx->d_sup_tmp, &ctx->d_sup_bits,
                     &ctx->d_sup_miss, &ctx->d_sup_len, &ctx->d_uns_seg, &ctx->d_uns_runcnt, &ctx->d_uns_misscnt, &ctx->d_uns_tmp,
                     &ctx->d_uns_runs, &ctx->d_uns_off };
  for (auto* b : bufs) b->release();
  if (ctx->l2_window_set) { cudaCtxResetPersistingL2Cache(); cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0); }
  for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : ctx->edit_ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : ctx->wave_ev) if (ev) cudaEventDestroy(ev);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

int gp_ctx_set_stream(gp_ctx* ctx, void* cuda_stream)
{
  if (!ctx) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return GP_OK;
}

int gp_ctx_synchronize(gp_ctx* ctx)
{
  if (!ctx) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return GP_OK;
}

// After an overlapped pass that kept SMs back for the edit kernel: did the build CTAs that left really come in whole
// SMs (the kernel counts them per %smid)?  Returns the number of SMs vacated; remembers a mismatch, after which
// gp_pipeline_run lets the two kernels share every SM again.  The stream must be idle.
static uint32_t sm_split_check(gp_ctx* ctx)
{
  if (!ctx->edit_sms || !ctx->d_sm_table.p) return 0;
  std::vector<uint32_t> t(1 + 2 * 2048);
  if (cudaMemcpy(t.data(), ctx->d_sm_table.p, t.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return 0; }
  uint32_t full = 0, other = 0, given_back = 0;
  const uint32_t keep = uint32_t(ctx->sm_count) - ctx->edit_sms;
  for (size_t i = 0; i < 2048; i++) {
    const uint32_t arrived = t[1 + 2 * i], rank_p1 = t[2 + 2 * i];
    if (arrived == ctx->edit_ctas_per_sm) { full++; if (rank_p1 > keep) given_back++; }
    else if (arrived) other++;
  }
  const bool ok = !other && full == uint32_t(ctx->sm_count) && given_back == ctx->edit_sms;
  if (ctx->sm_split_state == 0 || !ok) ctx->sm_split_state = ok ? 1 : -1;
  return ok ? given_back : 0;
}

int gp_get_stats(const gp_ctx* cctx, gp_stats* out)
{
  if (!cctx || !out) return GP_ERR_ARG;
  gp_ctx* ctx = const_cast<gp_ctx*>(cctx);
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->pack_timed) cudaEventElapsedTime(&ctx->stats.pack_ms, ctx->ev[0], ctx->ev[1]);
  if (ctx->build_timed && ctx->pipelined) {
    // overlapped pass: one span for both stages by events, the kernels' own spans from their device timers
    cudaEventElapsedTime(&ctx->stats.build_ms, ctx->ev[2], ctx->ev[3]);
    unsigned long long c[gp::kBuildCounters], pc[8];
    GP_CUDA(ctx, cudaMemcpy(c, ctx->d_counters.p, sizeof c, cudaMemcpyDeviceToHost));
    GP_CUDA(ctx, cudaMemcpy(pc, ctx->d_pcounters.p, sizeof pc, cudaMemcpyDeviceToHost));
    ctx->stats.kmer_ops = c[0];
    ctx->stats.serial_kmers = c[1];
    ctx->stats.build_kernel_ms = float(double(c[21] - c[20]) * 1e-6);
    ctx->stats.edit_kernel_ms = float(double(pc[5] - pc[4]) * 1e-6);
    ctx->stats.polish_ms = ctx->stats.edit_kernel_ms;
    ctx->stats.triggers = pc[0]; ctx->stats.edits = pc[1]; ctx->stats.masked = pc[2]; ctx->stats.rollbacks = pc[3];
    ctx->stats.edit_sms = sm_split_check(ctx); // SMs that were really vacated
    *out = ctx->stats;
    return GP_OK;
  }
  if (ctx->build_timed) {
    cudaEventElapsedTime(&ctx->stats.build_ms, ctx->ev[2], ctx->ev[3]);
    ctx->stats.build_kernel_ms = 0;
    for (size_t wv = 0; wv < ctx->wave_first.size() && 2 * wv + 1 < ctx->wave_ev.size(); wv++) {
      float t = 0;
      if (cudaEventElapsedTime(&t, ctx->wave_ev[2 * wv], ctx->wave_ev[2 * wv + 1]) == cudaSuccess) ctx->stats.build_kernel_ms += t;
    }
    unsigned long long c[2] = { 0, 0 };
    GP_CUDA(ctx, cudaMemcpy(c, ctx->d_counters.p, sizeof c, cudaMemcpyDeviceToHost));
    ctx->stats.kmer_ops = c[0];
    ctx->stats.serial_kmers = c[1];
  }
  if (ctx->polish_timed && ctx->edit_ev_valid) { // (a pipelined polish has no events of its own)
    cudaEventElapsedTime(&ctx->stats.polish_ms, ctx->ev[4], ctx->ev[5]);
    ctx->stats.edit_kernel_ms = 0;
    if (ctx->n_contigs) cudaEventElapsedTime(&ctx->stats.edit_kernel_ms, ctx->edit_ev[0], ctx->edit_ev[1]);
    unsigned long long c[4] = { 0, 0, 0, 0 };
    GP_CUDA(ctx, cudaMemcpy(c, ctx->d_pcounters.p, sizeof c, cudaMemcpyDeviceToHost));
    ctx->stats.triggers = c[0]; ctx->stats.edits = c[1]; ctx->stats.masked = c[2]; ctx->stats.rollbacks = c[3];
  }
  *out = ctx->stats;
  return GP_OK;
}

// ------------------------------------------------------------------------------------
// read store
// ------------------------------------------------------------------------------------
// The store is laid out from the read lengths alone; the bases then arrive in slabs, are packed on the device
// (2 bits + 1 mask bit per base) and the ASCII staging is reused: the device never holds more than
// kReadSlabBytes (or the longest read) of ASCII next to the packed store (0.375 B/base).
static const uint64_t kReadSlabBytes = 256ull << 20;

int gp_reads_begin(gp_ctx* ctx, uint64_t n_reads, const uint32_t* lens)
{
  if (!ctx || (!lens && n_reads)) return GP_ERR_ARG;
  if (n_reads > 0xFFFFFFF0ull) GP_FAIL(ctx, GP_ERR_ARG, "too many reads");
  cudaSetDevice(ctx->cfg.device);
  ctx->n_reads = 0;
  ctx->reads_next = 0;
  ctx->h_read_len.assign(lens, lens + n_reads);
  ctx->h_read_boff.resize(n_reads + 1);
  uint64_t b = 0, longest = 0;
  for (uint64_t r = 0; r < n_reads; r++) {
    if (lens[r] >= (1u << 31)) GP_FAIL(ctx, GP_ERR_ARG, "read longer than 2^31 bases");
    ctx->h_read_boff[r] = b;
    b += (uint64_t(lens[r]) + 31) & ~31ull;
    longest = std::max<uint64_t>(longest, lens[r]);
  }
  ctx->h_read_boff[n_reads] = b;
  const uint64_t words = b / 32 + 2; // one spare word past the last read for the window loads
  ctx->read_slab = std::max(kReadSlabBytes, longest);
  if (const char* e = std::getenv("GP_READ_SLAB_BYTES")) ctx->read_slab = std::max<uint64_t>(uint64_t(std::atoll(e)), std::max<uint64_t>(longest, 1));
  GP_CUDA(ctx, ctx->d_read_boff.ensure((n_reads + 1) * 8));
  GP_CUDA(ctx, ctx->d_read_len.ensure((n_reads + 1) * 4));
  GP_CUDA(ctx, ctx->d_pk.ensure(words * 8));
  GP_CUDA(ctx, ctx->d_nm.ensure(words * 4));
  cudaStream_t s = ctx->stream;
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_read_boff.p, ctx->h_read_boff.data(), (n_reads + 1) * 8, cudaMemcpyHostToDevice, s));
  if (n_reads) GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_read_len.p, ctx->h_read_len.data(), n_reads * 4, cudaMemcpyHostToDevice, s));
  // the two spare words must read as "no seed"
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_nm.as<uint32_t>() + (words - 2), 0xFF, 8, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_pk.as<uint64_t>() + (words - 2), 0, 16, s));
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[0], s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  ctx->reads_total = n_reads;
  ctx->stats.pack_launches = 0;
  return GP_OK;
}

int gp_reads_append(gp_ctx* ctx, const char* seqs, uint64_t n)
{
  if (!ctx || (!seqs && n)) return GP_ERR_ARG;
  if (ctx->reads_next + n > ctx->reads_total) GP_FAIL(ctx, GP_ERR_STATE, "gp_reads_append: more reads than gp_reads_begin announced");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t s = ctx->stream;
  uint64_t r = ctx->reads_next, done = 0; // `done` = bytes of seqs consumed
  const uint64_t r_end = r + n;
  std::vector<uint64_t> aoff;
  while (r < r_end) {
    // a slab: as many whole reads as fit (at least one)
    uint64_t r1 = r, bytes = 0;
    while (r1 < r_end && (r1 == r || bytes + ctx->h_read_len[r1] <= ctx->read_slab)) bytes += ctx->h_read_len[r1++];
    const uint64_t cnt = r1 - r;
    aoff.resize(cnt + 1);
    aoff[0] = 0;
    for (uint64_t i = 0; i < cnt; i++) aoff[i + 1] = aoff[i] + ctx->h_read_len[r + i];
    GP_CUDA(ctx, ctx->d_ascii.ensure(bytes + 16));
    GP_CUDA(ctx, ctx->d_ascii_off.ensure((cnt + 1) * 8));
    if (bytes) GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_ascii.p, seqs + done, bytes, cudaMemcpyHostToDevice, s));
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_ascii_off.p, aoff.data(), (cnt + 1) * 8, cudaMemcpyHostToDevice, s));
    gp::launch_pack_reads(ctx->d_ascii.as<char>(), ctx->d_ascii_off.as<uint64_t>(), ctx->d_read_boff.as<uint64_t>() + r,
                          ctx->d_pk.as<uint64_t>(), ctx->d_nm.as<uint32_t>(), uint32_t(cnt), s);
    GP_CUDA(ctx, cudaGetLastError());
    ctx->stats.pack_launches++;
    GP_CUDA(ctx, cudaStreamSynchronize(s)); // the staging buffers (device slab, host offsets) are reused by the next slab
    done += bytes;
    r = r1;
  }
  ctx->reads_next = r_end;
  return GP_OK;
}

int gp_reads_end(gp_ctx* ctx)
{
  if (!ctx) return GP_ERR_ARG;
  if (ctx->reads_next != ctx->reads_total) GP_FAIL(ctx, GP_ERR_STATE, "gp_reads_end: fewer reads appended than gp_reads_begin announced");
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->pack_timed = true;
  // the ASCII staging slab stays (the next upload reuses it) unless an extraordinarily long read blew it up
  if (ctx->d_ascii.cap > 2 * kReadSlabBytes) ctx->d_ascii.release();
  ctx->n_reads = ctx->reads_total;
  return GP_OK;
}

int gp_reads_upload(gp_ctx* ctx, const char* seqs, const uint64_t* offsets, uint64_t n_reads)
{
  if (!ctx || (!seqs && n_reads) || !offsets) return GP_ERR_ARG;
  std::vector<uint32_t> lens(n_reads);
  for (uint64_t r = 0; r < n_reads; r++) {
    const uint64_t len = offsets[r + 1] - offsets[r];
    if (len >= (1ull << 31)) GP_FAIL(ctx, GP_ERR_ARG, "read longer than 2^31 bases");
    lens[r] = uint32_t(len);
  }
  if (int rc = gp_reads_begin(ctx, n_reads, lens.data())) return rc;
  if (n_reads)
    if (int rc = gp_reads_append(ctx, seqs + offsets[0], n_reads)) return rc;
  return gp_reads_end(ctx);
}

// ------------------------------------------------------------------------------------
// filter build
// ------------------------------------------------------------------------------------
int gp_build_stage(gp_ctx* ctx, uint32_t n_batches, const uint64_t* batch_entry_off, const gp_read_entry* entries)
{
  if (!ctx || !batch_entry_off || (!entries && n_batches && batch_entry_off[n_batches])) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  const gp_config& c = ctx->cfg;
  const uint64_t n_entries = batch_entry_off[n_batches];
  std::vector<uint64_t> work(n_batches, 0);
  for (uint32_t b = 0; b < n_batches; b++) {
    for (uint64_t e = batch_entry_off[b]; e < batch_entry_off[b + 1]; e++) {
      if (entries[e].read_id >= ctx->n_reads) GP_FAIL(ctx, GP_ERR_ARG, "read_id out of range (upload reads first)");
      if (entries[e].kmer_threshold < 4) // fill_bfs, src/utils.cpp:105-107
        GP_FAIL(ctx, GP_ERR_ARG, "kmer_threshold must be greater than or equal to 4");
      work[b] += ctx->h_read_len[entries[e].read_id];
    }
  }
  // level-synchronous form: steps (32 k-mer starts) before every entry, per k; largest threshold per batch
  {
    std::vector<uint32_t> pre(size_t(c.nk) * (n_entries + 1), 0u), maxthr(std::max<uint32_t>(n_batches, 1), 0u);
    bool ok = true;
    uint64_t max_steps = 0;
    for (uint32_t ki = 0; ki < c.nk; ki++) {
      uint32_t* pk = pre.data() + size_t(ki) * (n_entries + 1);
      uint64_t acc = 0;
      for (uint64_t e = 0; e < n_entries; e++) {
        pk[e] = uint32_t(acc);
        const uint32_t len = ctx->h_read_len[entries[e].read_id];
        if (len >= c.k[ki]) acc += (uint64_t(len) - c.k[ki] + 1 + 31) / 32;
      }
      pk[n_entries] = uint32_t(acc);
      if (acc >= 0xFFFFFFFFull) ok = false;
      for (uint32_t b = 0; b < n_batches && ok; b++) {
        const uint64_t st = uint64_t(pk[batch_entry_off[b + 1]]) - pk[batch_entry_off[b]];
        max_steps = std::max(max_steps, st);
        if (st * 32 >= (1ull << 26)) ok = false; // occurrence clock is 26 bits
      }
    }
    std::vector<uint16_t> entry_rel(std::max<uint64_t>(n_entries, 1), 0);
    for (uint32_t b = 0; b < n_batches; b++) {
      if (batch_entry_off[b + 1] - batch_entry_off[b] > 0xFFFFull) ok = false; // step -> entry anchors are 16 bits
      for (uint64_t e = batch_entry_off[b]; e < batch_entry_off[b + 1]; e++) {
        maxthr[b] = std::max(maxthr[b], entries[e].kmer_threshold);
        if (entries[e].kmer_threshold > 24) ok = false; // the levels of two streams in flight must fit the 6-bit epoch tags (the reference caps T at 13)
        entry_rel[e] = uint16_t(e - batch_entry_off[b]);
      }
    }
    ctx->h_empty_streams.clear();
    for (uint32_t ki = 0; ki < c.nk; ki++) {
      const uint32_t* pk = pre.data() + size_t(ki) * (n_entries + 1);
      for (uint32_t b = 0; b < n_batches; b++)
        if (pk[batch_entry_off[b + 1]] == pk[batch_entry_off[b]]) ctx->h_empty_streams.push_back(b * c.nk + ki);
    }
    ctx->anchor_stride = 1;
    for (uint32_t ki = 0; ki < c.nk; ki++)
      ctx->anchor_stride = std::max<uint64_t>(ctx->anchor_stride, uint64_t(pre[size_t(ki) * (n_entries + 1) + n_entries]) + 1);
    ctx->levels_ok = ok;
    ctx->h_pre = pre;
    ctx->h_maxthr = maxthr;
    ctx->h_batch_entry_off.assign(batch_entry_off, batch_entry_off + n_batches + 1);
    ctx->n_entries = uint32_t(n_entries);
    ctx->alive_words = uint32_t(max_steps + 1);
    ctx->level_time_bits = 16; // occurrence times of the longest stream must fit
    // GP_LEVEL_TIME_BITS=n (16..26): a higher floor, i.e. narrower epoch tags, so that small inputs reach the tag clears
    // of the level kernel (the output does not depend on the width)
    if (const char* f = std::getenv("GP_LEVEL_TIME_BITS")) ctx->level_time_bits = uint32_t(std::min(26, std::max(16, std::atoi(f))));
    while (ctx->level_time_bits < 26 && (max_steps * 32) >> ctx->level_time_bits) ctx->level_time_bits++;
    GP_CUDA(ctx, ctx->d_step_pre.ensure(pre.size() * 4));
    GP_CUDA(ctx, ctx->d_batch_max_thr.ensure(maxthr.size() * 4));
    // level-synchronous kernel: two timestamp arrays alternate between the levels of the stream in flight; the LAST list
    // round of a stream (it only reads one of them) runs beside round 0 of the next (GP_LEVEL_OVERLAP=0: one stream at
    // a time, same arrays)
    ctx->level_slots = 2;
    if (const char* f = std::getenv("GP_LEVEL_OVERLAP")) ctx->level_slots = f[0] == '0' ? 1u : 2u;
    ctx->level_arrays = 2; // (three arrays let every late round be joined, but 120 MiB of timestamps do not stay in L2: 1.5x slower)
    if (const char* f = std::getenv("GP_LEVEL_ARRAYS")) ctx->level_arrays = f[0] == '3' ? 3u : 2u;
    GP_CUDA(ctx, ctx->d_V.ensure(gp::kCbfCounters * 4 * ctx->level_arrays));
    // warp-private survivor lists, kLevelSurvWords words per entry (a warp's region is its share of the steps,
    // rounded up, x 32), one buffer per stream in flight; then the barrier counter
    ctx->surv_cap = uint32_t(size_t(ctx->alive_words) * 32 + size_t(8192) * 9 * 32); // + (runs + 1) slack slots per warp
    GP_CUDA(ctx, ctx->d_alive.ensure(size_t(ctx->surv_cap) * gp::kLevelSurvWords * gp::kLevelListBufs * 4 + 64 + 8192));
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_step_pre.p, pre.data(), pre.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_batch_max_thr.p, maxthr.data(), maxthr.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (ok) {
      GP_CUDA(ctx, ctx->d_entry_rel.ensure(entry_rel.size() * 2));
      GP_CUDA(ctx, ctx->d_anchor.ensure(ctx->anchor_stride * c.nk * 2));
      GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_entry_rel.p, entry_rel.data(), entry_rel.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
      gp::launch_fill_anchor(ctx->d_step_pre.as<uint32_t>(), ctx->d_entry_rel.as<uint16_t>(), ctx->d_anchor.as<uint16_t>(),
                             uint32_t(n_entries), c.nk, ctx->anchor_stride, ctx->stream);
      GP_CUDA(ctx, cudaGetLastError());
    }
    GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  // which build kernel: 0 = auto (level-synchronous whenever the 26-bit occurrence clock suffices)
  {
    int algo = ctx->build_algo;
    if (const char* f = std::getenv("GP_BUILD_KERNEL")) algo = f[0] == 'l' ? 2 : (f[0] == 's' || f[0] == 'p') ? 1 : algo;
    if (algo == 0) algo = 2;
    if (!ctx->levels_ok) algo = 1;
    ctx->build_algo_resolved = algo;
  }
  const bool uses_cbf = ctx->build_algo_resolved == 1 || c.keep_counters;
  // Residency.  Filters (nk x 512 KiB per batch): all batches of the call when they fit and max_resident_filters allows
  // it; otherwise the pool holds one wave and is reused wave after wave (gp_pipeline_run polishes a wave before its
  // filters go, gp_build_output_host receives the payloads).  Counting filters (nk x 10 MiB per batch, in-order kernel
  // and keep_counters only) are always per wave.
  const uint64_t per_batch = uint64_t(c.nk) * gp::kCbfCounters, per_batch_bf = uint64_t(c.nk) * gp::kBfBytes;
  uint32_t wave = n_batches;
  if (c.max_resident_batches) wave = std::min(wave, c.max_resident_batches);
  {
    size_t free_b = 0, total_b = 0;
    GP_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
    const uint64_t usable = uint64_t(free_b) + ctx->d_cbf_pool.cap + ctx->d_bf_pool.cap;
    const uint64_t headroom = 3ull << 30;
    uint64_t bf_limit = n_batches;
    if (c.max_resident_filters) bf_limit = std::min<uint64_t>(bf_limit, c.max_resident_filters);
    // the pool may take up to half of what is free (the polish buffers and the lists come after it)
    const uint64_t fit_bf = usable > headroom ? (usable - headroom) / 2 / per_batch_bf : 0;
    if (fit_bf == 0 && n_batches) GP_FAIL(ctx, GP_ERR_OOM, "not enough device memory for one batch of filters");
    bf_limit = std::min(bf_limit, fit_bf);
    ctx->bf_all_resident = bf_limit >= n_batches;
    if (!ctx->bf_all_resident) wave = uint32_t(std::min<uint64_t>(wave, bf_limit));
    if (uses_cbf) {
      const uint64_t left = usable > headroom ? usable - headroom - (ctx->bf_all_resident ? uint64_t(n_batches) * per_batch_bf : 0) : 0;
      const uint64_t fit = left / (per_batch + (ctx->bf_all_resident ? 0 : per_batch_bf));
      if (fit == 0 && n_batches) GP_FAIL(ctx, GP_ERR_OOM, "not enough device memory for one batch of counting filters");
      wave = uint32_t(std::min<uint64_t>(wave, fit));
    }
  }
  GP_CUDA(ctx, ctx->d_bf_pool.ensure(std::max<uint64_t>(uint64_t(ctx->bf_all_resident ? n_batches : wave) * per_batch_bf, 4)));
  if (n_batches && uses_cbf) {
    cudaError_t e = ctx->d_cbf_pool.ensure(uint64_t(wave) * per_batch);
    while (e != cudaSuccess && wave > 1) { cudaGetLastError(); wave = (wave + 1) / 2; e = ctx->d_cbf_pool.ensure(uint64_t(wave) * per_batch); }
    GP_CUDA(ctx, e);
  }
  ctx->wave_batches = wave;
  ctx->wave_first.clear(); ctx->wave_count.clear(); ctx->wave_order_off.clear();
  std::vector<uint32_t> order_all;
  order_all.reserve(size_t(n_batches) * c.nk);
  for (uint32_t first = 0; first < n_batches; first += wave) {
    const uint32_t cnt = std::min(wave, n_batches - first);
    ctx->wave_first.push_back(first);
    ctx->wave_count.push_back(cnt);
    ctx->wave_order_off.push_back(uint32_t(order_all.size()));
    // longest stream first (the tail of the launch is one warp finishing one stream)
    std::vector<uint32_t> idx(size_t(cnt) * c.nk);
    std::iota(idx.begin(), idx.end(), 0u);
    std::stable_sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b2) {
      return work[first + a / c.nk] > work[first + b2 / c.nk];
    });
    order_all.insert(order_all.end(), idx.begin(), idx.end());
  }
  const size_t n_waves = ctx->wave_first.size();
  GP_CUDA(ctx, ctx->d_batch_entry_off.ensure((size_t(n_batches) + 1) * 8));
  GP_CUDA(ctx, ctx->d_entries.ensure(std::max<size_t>(n_entries, 1) * sizeof(gp_read_entry)));
  GP_CUDA(ctx, ctx->d_stream_order.ensure(std::max<size_t>(order_all.size(), 1) * 4));
  GP_CUDA(ctx, ctx->d_next.ensure(std::max<size_t>(n_waves, 1) * 4));
  GP_CUDA(ctx, ctx->d_counters.ensure(gp::kBuildCounters * 8));
  cudaStream_t s = ctx->stream;
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_batch_entry_off.p, batch_entry_off, (size_t(n_batches) + 1) * 8, cudaMemcpyHostToDevice, s));
  if (n_entries)
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_entries.p, entries, n_entries * sizeof(gp_read_entry), cudaMemcpyHostToDevice, s));
  if (!order_all.empty())
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_stream_order.p, order_all.data(), order_all.size() * 4, cudaMemcpyHostToDevice, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s)); // order_all is a local
  ctx->n_batches = n_batches;
  ctx->build_staged = true;
  ctx->filters_ready = false;
  ctx->build_done = false;
  return GP_OK;
}

// per stream, in launch order: steps, largest thr, batch (the level kernel reads it one stream ahead); build_order:
// the batches of a wave in gp_pipeline_run's order (h_batch_order)
static int build_stream_tab(gp_ctx* ctx, cudaStream_t s, bool build_order)
{
  const gp_config& c = ctx->cfg;
  const size_t total = size_t(ctx->n_batches) * c.nk;
  ctx->h_stream_tab.resize(std::max<size_t>(total, 1));
  const size_t ne1 = size_t(ctx->n_entries) + 1;
  size_t w = 0;
  for (size_t wv = 0; wv < ctx->wave_first.size(); wv++)
    for (uint32_t st = 0; st < ctx->wave_count[wv] * c.nk; st++, w++) {
      const uint32_t lb = st / c.nk, ki = st - lb * c.nk;
      const uint32_t b = build_order ? ctx->h_batch_order[ctx->wave_first[wv] + lb] : ctx->wave_first[wv] + lb;
      const uint32_t* pk = ctx->h_pre.data() + size_t(ki) * ne1;
      const uint32_t steps = pk[ctx->h_batch_entry_off[b + 1]] - pk[ctx->h_batch_entry_off[b]];
      ctx->h_stream_tab[w] = make_uint4(steps, ctx->h_maxthr[b] - 2u + ki, b, 0u);
    }
  GP_CUDA(ctx, ctx->d_stream_tab.ensure(ctx->h_stream_tab.size() * sizeof(uint4)));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_stream_tab.p, ctx->h_stream_tab.data(), ctx->h_stream_tab.size() * sizeof(uint4), cudaMemcpyHostToDevice, s));
  return GP_OK;
}

// pool slot of every batch when the pool holds one wave at a time: its position inside its wave (waves are uniform
// runs of wave_batches positions of the launch order)
static int upload_bf_slots(gp_ctx* ctx, cudaStream_t s, bool build_order)
{
  if (ctx->bf_all_resident) return GP_OK;
  const uint32_t nb = ctx->n_batches, wave = std::max(ctx->wave_batches, 1u);
  ctx->h_bf_slot.resize(nb);
  for (uint32_t pos = 0; pos < nb; pos++) ctx->h_bf_slot[build_order ? ctx->h_batch_order[pos] : pos] = pos % wave;
  GP_CUDA(ctx, ctx->d_bf_slot.ensure(std::max<size_t>(nb, 1) * 4));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bf_slot.p, ctx->h_bf_slot.data(), size_t(nb) * 4, cudaMemcpyHostToDevice, s));
  return GP_OK;
}

// level-synchronous build of wave wv on stream s (build_stream_tab first); batch_done / ctas_per_sm are
// gp_pipeline_run's (NULL, 0 otherwise)
static int build_launch_levels_wave(gp_ctx* ctx, cudaStream_t s, size_t wv, uint32_t* batch_done, int ctas_per_sm, uint32_t reserve_sms = 0)
{
  const gp_config& c = ctx->cfg;
  {
    size_t tab_off = 0;
    for (size_t i = 0; i < wv; i++) tab_off += size_t(ctx->wave_count[i]) * c.nk;
    // level-synchronous: all SMs on one stream at a time, timestamps resident in L2
    gp::LevelParams p;
    std::memset(&p, 0, sizeof p);
    p.pk = ctx->d_pk.as<uint64_t>();
    p.nm = ctx->d_nm.as<uint32_t>();
    p.read_boff = ctx->d_read_boff.as<uint64_t>();
    p.read_len = ctx->d_read_len.as<uint32_t>();
    p.batch_entry_off = ctx->d_batch_entry_off.as<uint64_t>();
    p.entries = ctx->d_entries.as<gp_read_entry>();
    p.step_pre = ctx->d_step_pre.as<uint32_t>();
    p.batch_max_thr = ctx->d_batch_max_thr.as<uint32_t>();
    p.anchor = ctx->d_anchor.as<uint16_t>();
    p.anchor_stride = ctx->anchor_stride;
    p.V = ctx->d_V.as<uint32_t>();
    p.surv = ctx->d_alive.as<uint32_t>();
    p.bars = reinterpret_cast<unsigned long long*>(ctx->d_alive.as<uint32_t>() + size_t(gp::kLevelSurvWords) * gp::kLevelListBufs * ctx->surv_cap);
    p.overlap = ctx->level_slots > 1 ? 1u : 0u;
    p.arrays = ctx->level_arrays;
    p.time_bits = ctx->level_time_bits;
    if (const char* f = std::getenv("GP_LEVEL_REPORT_CTA")) p.report_cta = uint32_t(std::atoi(f));
    p.cbf_pool = c.keep_counters ? ctx->d_cbf_pool.as<uint8_t>() : nullptr;
    p.bf_pool = ctx->d_bf_pool.as<uint32_t>();
    p.bf_slot = ctx->bf_all_resident ? nullptr : ctx->d_bf_slot.as<uint32_t>();
    p.counters = ctx->d_counters.as<unsigned long long>();
    p.surv_cap = ctx->surv_cap;
    p.n_entries = ctx->n_entries;
    p.n_streams = ctx->wave_count[wv] * c.nk;
    p.first_batch = ctx->wave_first[wv];
    p.stream_tab = ctx->d_stream_tab.as<uint4>() + tab_off;
    p.nk = c.nk;
    for (uint32_t i = 0; i < gp::kMaxK; i++) p.k[i] = i < c.nk ? c.k[i] : 0;
    if (c.keep_counters) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_cbf_pool.p, 0, uint64_t(p.n_streams) * gp::kCbfCounters, s));
    GP_CUDA(ctx, cudaMemsetAsync(ctx->d_V.p, 0xFF, gp::kCbfCounters * 4 * ctx->level_arrays, s));
    GP_CUDA(ctx, cudaMemsetAsync(p.bars, 0, 64 + 8192, s));
    p.speed = reinterpret_cast<uint32_t*>(p.bars + 8);
    {
      const char* e = std::getenv("GP_LEVEL_WEIGHTED");
      p.weighted = !(e && e[0] == '0') ? 1u : 0u;
    }
    while (ctx->wave_ev.size() < 2 * (wv + 1)) { cudaEvent_t e2 = nullptr; cudaEventCreate(&e2); ctx->wave_ev.push_back(e2); }
    if (!batch_done) GP_CUDA(ctx, cudaEventRecord(ctx->wave_ev[2 * wv], s));
    p.batch_done = batch_done;
    p.n_batches_total = ctx->n_batches;
    p.bf_host = ctx->bf_host_dev;
    // the timestamp arrays are the kernel's random-access working set: keep them in the persisting part of L2
    // (79 of 126 MiB on B200), so that the survivor lists, the sequence and the filters streaming through do not
    // evict them (+6 % k-mer ops/s).  Only when the window can cover them.
    {
      const size_t vbytes = gp::kCbfCounters * 4 * p.arrays;
      const char* e = std::getenv("GP_L2_PERSIST");
      const bool want = !(e && e[0] == '0') && ctx->l2_persist_max > 0 && vbytes <= size_t(ctx->l2_window_max);
      cudaStreamAttrValue av;
      std::memset(&av, 0, sizeof av);
      if (want) {
        // GP_L2_WINDOW=c: only the T_1 array (the densest one: every occurrence touches it twice), all of it
        const char* wsel = std::getenv("GP_L2_WINDOW");
        const bool only_c = wsel && wsel[0] == 'c' && p.arrays == 3u;
        const size_t wbytes = only_c ? gp::kCbfCounters * 4 : vbytes;
        av.accessPolicyWindow.base_ptr = only_c ? static_cast<void*>(ctx->d_V.as<uint32_t>() + 2 * gp::kCbfCounters) : ctx->d_V.p;
        av.accessPolicyWindow.num_bytes = wbytes;
        av.accessPolicyWindow.hitRatio = std::min(1.0f, float(ctx->l2_persist_max) / float(wbytes));
        av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
      } // else: an empty window switches the policy off
      if (want != ctx->l2_window_set) {
        // the set-aside is carved out of the normal L2: claim it only while the window uses it
        if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want ? size_t(ctx->l2_persist_max) : 0) != cudaSuccess) cudaGetLastError();
        if (!want) cudaCtxResetPersistingL2Cache();
      }
      if (want || ctx->l2_window_set) {
        GP_CUDA(ctx, cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &av));
        ctx->l2_window_set = want;
      }
    }
    if (std::getenv("GP_LEVEL_CTA_TIMES")) { // diagnostics of every CTA (gp_build_cta_times)
      GP_CUDA(ctx, ctx->d_cta_times.ensure(size_t(ctx->sm_count) * 4 * 32 * 8));
      GP_CUDA(ctx, cudaMemsetAsync(ctx->d_cta_times.p, 0, size_t(ctx->sm_count) * 4 * 32 * 8, s));
      p.cta_times = ctx->d_cta_times.as<unsigned long long>();
    }
    if (reserve_sms) { // the launch fills every SM; the CTAs of the last `reserve_sms` SMs leave at once (see the kernel)
      const size_t bytes = (1 + 2 * 2048) * 4; // (%nsmid is far below 2048)
      GP_CUDA(ctx, ctx->d_sm_table.ensure(bytes));
      GP_CUDA(ctx, cudaMemsetAsync(ctx->d_sm_table.p, 0, bytes, s));
      p.keep_sms = uint32_t(ctx->sm_count) - reserve_sms;
      p.sm_table = ctx->d_sm_table.as<uint32_t>();
    }
    ctx->level_grid = uint32_t((ctx->sm_count - int(reserve_sms)) * gp::levels_ctas_per_sm(ctas_per_sm));
    GP_CUDA(ctx, gp::launch_build_filters_levels(p, ctx->sm_count, s, ctas_per_sm));
    if (!batch_done) GP_CUDA(ctx, cudaEventRecord(ctx->wave_ev[2 * wv + 1], s));
  }
  return GP_OK;
}

// in-order kernel (one warp per stream, counters in HBM), wave wv
static int build_launch_inorder_wave(gp_ctx* ctx, cudaStream_t s, size_t wv)
{
  const gp_config& c = ctx->cfg;
  gp::BuildParams p;
  std::memset(&p, 0, sizeof p);
  p.pk = ctx->d_pk.as<uint64_t>();
  p.nm = ctx->d_nm.as<uint32_t>();
  p.read_boff = ctx->d_read_boff.as<uint64_t>();
  p.read_len = ctx->d_read_len.as<uint32_t>();
  p.batch_entry_off = ctx->d_batch_entry_off.as<uint64_t>();
  p.entries = ctx->d_entries.as<gp_read_entry>();
  p.cbf_pool = ctx->d_cbf_pool.as<uint8_t>();
  p.bf_pool = ctx->d_bf_pool.as<uint32_t>();
  p.bf_slot = ctx->bf_all_resident ? nullptr : ctx->d_bf_slot.as<uint32_t>();
  p.stream_order = ctx->d_stream_order.as<uint32_t>() + ctx->wave_order_off[wv];
  p.next_stream = ctx->d_next.as<uint32_t>() + wv;
  p.counters = ctx->d_counters.as<unsigned long long>();
  p.n_streams = ctx->wave_count[wv] * c.nk;
  p.first_batch = ctx->wave_first[wv];
  p.nk = c.nk;
  for (uint32_t i = 0; i < gp::kMaxK; i++) p.k[i] = i < c.nk ? c.k[i] : 0;
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_cbf_pool.p, 0, uint64_t(p.n_streams) * gp::kCbfCounters, s));
  while (ctx->wave_ev.size() < 2 * (wv + 1)) { cudaEvent_t e2 = nullptr; cudaEventCreate(&e2); ctx->wave_ev.push_back(e2); }
  GP_CUDA(ctx, cudaEventRecord(ctx->wave_ev[2 * wv], s));
  gp::launch_build_filters(p, ctx->sm_count, s);
  GP_CUDA(ctx, cudaGetLastError());
  GP_CUDA(ctx, cudaEventRecord(ctx->wave_ev[2 * wv + 1], s));
  return GP_OK;
}

// a wave's filters are final on the device and the pool is about to be reused: hand the payloads over (the level
// kernel has streamed them to the named host buffer itself; the in-order kernel has not)
static int wave_payloads_out(gp_ctx* ctx, cudaStream_t s, size_t wv, bool kernel_streams)
{
  if (ctx->bf_all_resident || kernel_streams || !ctx->bf_host_user) return GP_OK;
  const uint64_t per = uint64_t(ctx->cfg.nk) * gp::kBfBytes;
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->bf_host_user + uint64_t(ctx->wave_first[wv]) * per, ctx->d_bf_pool.p,
                               uint64_t(ctx->wave_count[wv]) * per, cudaMemcpyDeviceToHost, s));
  return GP_OK;
}

int gp_build_run(gp_ctx* ctx)
{
  if (!ctx) return GP_ERR_ARG;
  if (!ctx->build_staged) GP_FAIL(ctx, GP_ERR_STATE, "gp_build_run before gp_build_stage");
  cudaSetDevice(ctx->cfg.device);
  const gp_config& c = ctx->cfg;
  cudaStream_t s = ctx->stream;
  if (!ctx->bf_all_resident && !ctx->bf_host_user)
    GP_FAIL(ctx, GP_ERR_STATE, "the filters of this call are not all resident at once (max_resident_filters / device memory): "
                               "name a page-locked destination with gp_build_output_host, or use gp_pipeline_run");
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[2], s));
  ctx->pipelined = false;
  uint32_t launches = 0;
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, gp::kBuildCounters * 8, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.as<unsigned long long>() + 20, 0xFF, 8, s)); // first start time: atomicMin
  const uint64_t per_bf = uint64_t(c.nk) * gp::kBfBytes;
  if (ctx->n_batches) {
    GP_CUDA(ctx, cudaMemsetAsync(ctx->d_next.p, 0, ctx->wave_first.size() * 4, s));
    if (ctx->bf_all_resident) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_bf_pool.p, 0, uint64_t(ctx->n_batches) * per_bf, s));
  }
  const int algo = ctx->build_algo_resolved;
  if (int rc = upload_bf_slots(ctx, s, false)) return rc;
  if (algo == 2)
    if (int rc = build_stream_tab(ctx, s, false)) return rc;
  for (size_t wv = 0; wv < ctx->wave_first.size(); wv++) {
    if (!ctx->bf_all_resident) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_bf_pool.p, 0, uint64_t(ctx->wave_count[wv]) * per_bf, s));
    if (algo == 2) { if (int rc = build_launch_levels_wave(ctx, s, wv, nullptr, 0)) return rc; }
    else if (int rc = build_launch_inorder_wave(ctx, s, wv)) return rc;
    if (int rc = wave_payloads_out(ctx, s, wv, algo == 2 && ctx->bf_host_dev)) return rc;
    launches += 1;
  }
  // the named host buffer holds every payload after this run: written by the level kernel itself, or wave by wave
  ctx->bf_streamed = ctx->bf_host_user && ((algo == 2 && ctx->bf_host_dev) || !ctx->bf_all_resident);
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[3], s));
  ctx->build_timed = true;
  ctx->stats.build_launches = launches;
  ctx->stats.build_kernel = uint32_t(algo);
  ctx->stats.build_slots = algo == 2 ? ctx->level_slots : 0;
  ctx->stats.level_time_bits = algo == 2 ? ctx->level_time_bits : 0;
  ctx->filters_ready = ctx->bf_all_resident; // (a later gp_polish needs them all)
  ctx->build_done = true;
  return GP_OK;
}

int gp_build_round_times(gp_ctx* ctx, uint64_t out[32])
{
  if (!ctx || !out) return GP_ERR_ARG;
  if (!ctx->build_done) GP_FAIL(ctx, GP_ERR_STATE, "no filters have been built");
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  unsigned long long c[gp::kBuildCounters];
  GP_CUDA(ctx, cudaMemcpy(c, ctx->d_counters.p, sizeof c, cudaMemcpyDeviceToHost));
  std::memset(out, 0, 32 * 8);
  for (uint32_t i = 0; i < gp::kLevelDiag; i++) out[i] = c[gp::kLevelDiagAt + i];
  out[31] = c[17];
  return GP_OK;
}

int gp_debug_nthash(gp_ctx* ctx, uint64_t read_id, uint32_t k, uint64_t* hashes, uint8_t* valid, uint64_t cap_positions,
                    uint64_t* n_positions)
{
  if (!ctx || !hashes || !valid || !n_positions) return GP_ERR_ARG;
  if (read_id >= ctx->n_reads) GP_FAIL(ctx, GP_ERR_ARG, "read_id out of range (upload reads first)");
  if (k < 4 || k > 32) GP_FAIL(ctx, GP_ERR_ARG, "k must be within 4..32");
  cudaSetDevice(ctx->cfg.device);
  const uint32_t len = ctx->h_read_len[read_id];
  const uint64_t npos = len >= k ? uint64_t(len) - k + 1 : 0;
  *n_positions = npos;
  if (npos == 0) return GP_OK;
  if (npos > cap_positions) GP_FAIL(ctx, GP_ERR_ARG, "gp_debug_nthash: output too small (needed positions are in n_positions)");
  uint64_t boff = 0;
  GP_CUDA(ctx, cudaMemcpy(&boff, ctx->d_read_boff.as<uint64_t>() + read_id, 8, cudaMemcpyDeviceToHost));
  DevBuf dh, dv;
  GP_CUDA(ctx, dh.ensure(npos * 32));
  cudaError_t e = dv.ensure(npos);
  if (e != cudaSuccess) { dh.release(); GP_CUDA(ctx, e); }
  gp::launch_debug_nthash(ctx->d_pk.as<uint64_t>(), ctx->d_nm.as<uint32_t>(), boff >> 5, len, k, dh.as<uint64_t>(), dv.as<uint8_t>(), ctx->stream);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(hashes, dh.p, npos * 32, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(valid, dv.p, npos, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  dh.release(); dv.release();
  GP_CUDA(ctx, e);
  return GP_OK;
}

int gp_build_cta_times(gp_ctx* ctx, uint64_t* out, uint32_t cap_ctas, uint32_t* n_ctas)
{
  if (!ctx || !out || !n_ctas) return GP_ERR_ARG;
  if (!ctx->build_done || !ctx->d_cta_times.p) GP_FAIL(ctx, GP_ERR_STATE, "no per-CTA times were recorded (set GP_LEVEL_CTA_TIMES=1 before the build)");
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *n_ctas = std::min(cap_ctas, ctx->level_grid);
  GP_CUDA(ctx, cudaMemcpy(out, ctx->d_cta_times.p, size_t(*n_ctas) * 32 * 8, cudaMemcpyDeviceToHost));
  return GP_OK;
}

void* gp_host_alloc(uint64_t bytes)
{
  void* p = nullptr;
  if (cudaHostAlloc(&p, size_t(bytes), cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}

void gp_host_free(void* p)
{
  if (p) cudaFreeHost(p);
}

int gp_build_output_host(gp_ctx* ctx, uint8_t* bf_out_pinned)
{
  if (!ctx) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  ctx->bf_host_user = nullptr;
  ctx->bf_host_dev = nullptr;
  ctx->bf_streamed = false;
  if (!bf_out_pinned) return GP_OK;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, bf_out_pinned) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
    cudaGetLastError();
    GP_FAIL(ctx, GP_ERR_ARG, "gp_build_output_host needs page-locked host memory (cudaHostAlloc / cudaHostRegister)");
  }
  ctx->bf_host_user = bf_out_pinned;
  ctx->bf_host_dev = static_cast<uint32_t*>(at.devicePointer);
  return GP_OK;
}

int gp_build_fetch(gp_ctx* ctx, uint8_t* bf_out)
{
  if (!ctx) return GP_ERR_ARG;
  if (!ctx->build_done && !ctx->filters_ready) GP_FAIL(ctx, GP_ERR_STATE, "no filters have been built");
  cudaSetDevice(ctx->cfg.device);
  if (bf_out && bf_out == ctx->bf_host_user && ctx->bf_streamed) {
    // every final filter is in this buffer already (written by the build kernel, or copied wave by wave); streams
    // without k-mers are zeros
    GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t sidx : ctx->h_empty_streams) std::memset(bf_out + uint64_t(sidx) * gp::kBfBytes, 0, gp::kBfBytes);
    return GP_OK;
  }
  if (bf_out && !ctx->bf_all_resident)
    GP_FAIL(ctx, GP_ERR_STATE, "the filters of earlier waves are no longer resident: their payloads went to the buffer named with "
                               "gp_build_output_host (pass that pointer)");
  if (bf_out && ctx->n_batches)
    GP_CUDA(ctx, cudaMemcpyAsync(bf_out, ctx->d_bf_pool.p, uint64_t(ctx->n_batches) * ctx->cfg.nk * gp::kBfBytes,
                                 cudaMemcpyDeviceToHost, ctx->stream));
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return GP_OK;
}

int gp_build_fetch_cbf(gp_ctx* ctx, uint32_t batch, uint32_t k_index, uint8_t* cbf_out)
{
  if (!ctx || !cbf_out) return GP_ERR_ARG;
  if (!ctx->build_done) GP_FAIL(ctx, GP_ERR_STATE, "no filters have been built");
  if (batch >= ctx->n_batches || k_index >= ctx->cfg.nk) GP_FAIL(ctx, GP_ERR_ARG, "batch / k index out of range");
  if (ctx->build_algo_resolved == 2 && !ctx->cfg.keep_counters)
    GP_FAIL(ctx, GP_ERR_STATE, "counting-filter bytes were not materialised: create the context with keep_counters = 1");
  // counting filters of a wave are overwritten by the next wave: only the last wave is still resident
  const size_t last = ctx->wave_first.size() - 1;
  if (batch < ctx->wave_first[last]) GP_FAIL(ctx, GP_ERR_STATE, "counting filter of an earlier wave is no longer resident");
  cudaSetDevice(ctx->cfg.device);
  const uint64_t sid = uint64_t(batch - ctx->wave_first[last]) * ctx->cfg.nk + k_index;
  GP_CUDA(ctx, cudaMemcpyAsync(cbf_out, ctx->d_cbf_pool.as<uint8_t>() + sid * gp::kCbfCounters, gp::kCbfCounters,
                               cudaMemcpyDeviceToHost, ctx->stream));
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return GP_OK;
}

int gp_build_filters(gp_ctx* ctx, uint32_t n_batches, const uint64_t* batch_entry_off, const gp_read_entry* entries,
                     uint8_t* bf_out)
{
  int rc = gp_build_stage(ctx, n_batches, batch_entry_off, entries);
  if (rc) return rc;
  if ((rc = gp_build_run(ctx))) return rc;
  return gp_build_fetch(ctx, bf_out);
}

int gp_filters_load(gp_ctx* ctx, uint32_t n_batches, const uint8_t* bf_payloads)
{
  if (!ctx || (!bf_payloads && n_batches)) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  const uint64_t bytes = uint64_t(n_batches) * ctx->cfg.nk * gp::kBfBytes;
  GP_CUDA(ctx, ctx->d_bf_pool.ensure(std::max<uint64_t>(bytes, 4)));
  if (bytes) GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bf_pool.p, bf_payloads, bytes, cudaMemcpyHostToDevice, ctx->stream));
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->n_batches = n_batches;
  ctx->filters_ready = true;
  ctx->bf_all_resident = true;
  ctx->build_staged = false;
  ctx->build_done = false;
  return GP_OK;
}

// ------------------------------------------------------------------------------------
// polish
// ------------------------------------------------------------------------------------
static int polish_layout(gp_ctx* ctx)
{
  const uint32_t n = ctx->n_contigs;
  const uint32_t g = ctx->grow;
  // GP_POLISH_CAPS="bytes,nodes" (either may be empty: the default): the first layout gives a contig len + bytes of
  // buffer and that many rope nodes, so that small inputs reach the overflow re-run of polish_settle
  int64_t caps[2] = {-1, -1};
  if (const char* f = std::getenv("GP_POLISH_CAPS")) {
    const char* comma = std::strchr(f, ',');
    if (f[0] && f[0] != ',') caps[0] = std::max(0ll, std::atoll(f));
    if (comma && comma[1]) caps[1] = std::max(1ll, std::atoll(comma + 1)); // (the root node is written unchecked)
  }
  ctx->h_cap_off.assign(n + 1, 0);
  ctx->h_node_off.assign(n + 1, 0);
  for (uint32_t i = 0; i < n; i++) {
    const uint64_t len = ctx->h_len[i];
    uint64_t cap = len + (caps[0] >= 0 ? uint64_t(caps[0]) : (len >> 1) + 4096);
    uint64_t nodes = caps[1] >= 0 ? uint64_t(caps[1]) : (len >> 2) + 2048;
    cap <<= g; nodes <<= g;
    cap = (cap + 15) & ~15ull;
    if (cap >= (1ull << 32)) { ctx->err = "contig too long for 32-bit positions"; return GP_ERR_ARG; }
    ctx->h_cap_off[i + 1] = ctx->h_cap_off[i] + cap;
    ctx->h_node_off[i + 1] = ctx->h_node_off[i] + nodes;
  }
  GP_CUDA(ctx, ctx->d_buf0.ensure(std::max<uint64_t>(ctx->h_cap_off[n], 16)));
  GP_CUDA(ctx, ctx->d_buf1.ensure(std::max<uint64_t>(ctx->h_cap_off[n], 16)));
  GP_CUDA(ctx, ctx->d_nodes.ensure(std::max<uint64_t>(ctx->h_node_off[n], 1) * sizeof(gp::EdNode)));
  if (ctx->cfg.track_edits) { // origins: 4 B per byte of capacity, same layout
    GP_CUDA(ctx, ctx->d_orig0.ensure(std::max<uint64_t>(ctx->h_cap_off[n], 16) * 4));
    GP_CUDA(ctx, ctx->d_orig1.ensure(std::max<uint64_t>(ctx->h_cap_off[n], 16) * 4));
  }
  GP_CUDA(ctx, ctx->d_cap_off.ensure((size_t(n) + 1) * 8));
  GP_CUDA(ctx, ctx->d_node_off.ensure((size_t(n) + 1) * 8));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_cap_off.p, ctx->h_cap_off.data(), (size_t(n) + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_node_off.p, ctx->h_node_off.data(), (size_t(n) + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return GP_OK;
}

int gp_polish_stage(gp_ctx* ctx, uint32_t n_contigs, const char* seqs, const uint64_t* offsets, const uint32_t* contig_batch)
{
  if (!ctx || !offsets || (!seqs && n_contigs && offsets[n_contigs]) || (!contig_batch && n_contigs)) return GP_ERR_ARG;
  if (!ctx->filters_ready && !ctx->build_staged)
    GP_FAIL(ctx, GP_ERR_STATE, "gp_polish needs filters (gp_build_filters, gp_build_stage or gp_filters_load)");
  cudaSetDevice(ctx->cfg.device);
  const uint32_t n = n_contigs;
  ctx->n_contigs = n;
  ctx->h_len.resize(n);
  ctx->h_in_off.assign(offsets, offsets + n + 1);
  ctx->h_batch.assign(contig_batch, contig_batch + n);
  for (uint32_t i = 0; i < n; i++) {
    const uint64_t len = offsets[i + 1] - offsets[i];
    if (len >= (1ull << 31)) GP_FAIL(ctx, GP_ERR_ARG, "contig longer than 2^31 bases");
    if (contig_batch[i] >= ctx->n_batches) GP_FAIL(ctx, GP_ERR_ARG, "contig_batch out of range of the current filter set");
    ctx->h_len[i] = uint32_t(len);
  }
  ctx->h_order.resize(n);
  std::iota(ctx->h_order.begin(), ctx->h_order.end(), 0u);
  std::stable_sort(ctx->h_order.begin(), ctx->h_order.end(), [&](uint32_t a, uint32_t b) { return ctx->h_len[a] > ctx->h_len[b]; });
  const uint64_t total = offsets[n];
  GP_CUDA(ctx, ctx->d_input.ensure(std::max<uint64_t>(total, 16)));
  GP_CUDA(ctx, ctx->d_in_off.ensure((size_t(n) + 1) * 8));
  GP_CUDA(ctx, ctx->d_cur_len.ensure(std::max<size_t>(n, 1) * 4));
  GP_CUDA(ctx, ctx->d_which.ensure(std::max<size_t>(n, 1)));
  GP_CUDA(ctx, ctx->d_dropped.ensure(std::max<size_t>(n, 1)));
  GP_CUDA(ctx, ctx->d_contig_batch.ensure(std::max<size_t>(n, 1) * 4));
  GP_CUDA(ctx, ctx->d_order.ensure(std::max<size_t>(n, 1) * 4));
  GP_CUDA(ctx, ctx->d_pnext.ensure(4));
  GP_CUDA(ctx, ctx->d_pcounters.ensure(64));
  GP_CUDA(ctx, ctx->d_error.ensure(4));
  cudaStream_t s = ctx->stream;
  if (total) GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_input.p, seqs, total, cudaMemcpyHostToDevice, s));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_in_off.p, offsets, (size_t(n) + 1) * 8, cudaMemcpyHostToDevice, s));
  if (n) {
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_contig_batch.p, contig_batch, size_t(n) * 4, cudaMemcpyHostToDevice, s));
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_order.p, ctx->h_order.data(), size_t(n) * 4, cudaMemcpyHostToDevice, s));
  }
  ctx->grow = 0;
  if (int rc = polish_layout(ctx)) return rc;
  ctx->polish_staged = true;
  ctx->polish_done = false;
  ctx->edits_polish = false;
  ctx->support_polish = false;
  return GP_OK;
}

// counters + contigs into their working buffers (stream s)
static int polish_prepare(gp_ctx* ctx)
{
  cudaStream_t s = ctx->stream;
  const uint32_t n = ctx->n_contigs;
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_pnext.p, 0, 4, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_pcounters.p, 0, 64, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_pcounters.as<unsigned long long>() + 4, 0xFF, 8, s)); // first start time: atomicMin
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_error.p, 0, 4, s));
  if (n == 0) return GP_OK;
  const uint32_t grid = std::min<uint32_t>(n, uint32_t(ctx->sm_count) * 8u);
  uint32_t* orig0 = ctx->cfg.track_edits ? ctx->d_orig0.as<uint32_t>() : nullptr;
  scatter_contigs_kernel<<<grid, 256, 0, s>>>(ctx->d_input.as<char>(), ctx->d_in_off.as<uint64_t>(), ctx->d_buf0.as<char>(),
                                              ctx->d_cap_off.as<uint64_t>(), ctx->d_cur_len.as<uint32_t>(), orig0, n);
  GP_CUDA(ctx, cudaGetLastError());
  return GP_OK;
}

// the edit kernel on stream es (the context's stream unless pipelined: then `order`, `batch_done` and
// alongside are gp_pipeline_run's)
static int polish_edit(gp_ctx* ctx, cudaStream_t es, const uint32_t* order, uint32_t n_order, const uint32_t* batch_done, int alongside)
{
  const gp_config& c = ctx->cfg;
  const uint32_t n = order ? n_order : ctx->n_contigs; // slots of `order` this launch works through
  if (n == 0) return GP_OK;
  gp::EditParams p;
  std::memset(&p, 0, sizeof p);
  p.n_contigs = n;
  p.buf[0] = ctx->d_buf0.as<char>();
  p.buf[1] = ctx->d_buf1.as<char>();
  p.cap_off = ctx->d_cap_off.as<uint64_t>();
  p.cur_len = ctx->d_cur_len.as<uint32_t>();
  p.which = ctx->d_which.as<uint8_t>();
  p.dropped = ctx->d_dropped.as<uint8_t>();
  p.nodes = ctx->d_nodes.as<gp::EdNode>();
  p.node_off = ctx->d_node_off.as<uint64_t>();
  p.contig_batch = ctx->d_contig_batch.as<uint32_t>();
  p.bf_pool = ctx->d_bf_pool.as<uint32_t>();
  p.bf_slot = ctx->bf_all_resident ? nullptr : ctx->d_bf_slot.as<uint32_t>();
  p.order = order ? order : ctx->d_order.as<uint32_t>();
  p.batch_done = batch_done;
  p.n_batches = ctx->n_batches;
  p.next_contig = ctx->d_pnext.as<uint32_t>();
  p.counters = ctx->d_pcounters.as<unsigned long long>();
  p.error = ctx->d_error.as<int>();
  p.nk = c.nk;
  for (uint32_t i = 0; i < c.nk; i++) {
    p.k[i] = c.k[i];
    // the reference's float expressions, evaluated once on the host
    // (ntedit.cpp:1521-1523, 1624-1626 / 1335-1337, 1228-1230, 2024-2025)
    const float kf = static_cast<float>(c.k[i]);
    const float jf = static_cast<float>(c.jump);
    if (c.use_ratio) {
      p.thr_missing[i] = (kf / jf) * c.missing_ratio;
      p.thr_edit[i] = (kf / jf) * c.edit_ratio;
      p.thr_del[i] = (1 + (kf / jf)) * c.edit_ratio;
    } else { // -x / -y form (ntedit.cpp:1519-1520, 1622-1623, 1333-1334, 1226-1227)
      p.thr_missing[i] = kf / c.missing_threshold;
      p.thr_edit[i] = kf / c.edit_threshold;
      p.thr_del[i] = kf / c.edit_threshold;
    }
    p.insertion_cap[i] = static_cast<unsigned>(kf * 1.5f);
  }
  p.max_insertions = c.max_insertions; p.max_deletions = c.max_deletions; p.jump = c.jump;
  p.min_contig_len = c.min_contig_len; p.mode = c.mode; p.mask = c.mask;
  if (c.track_edits) {
    p.orig[0] = ctx->d_orig0.as<uint32_t>();
    p.orig[1] = ctx->d_orig1.as<uint32_t>();
  }
  if (!alongside) GP_CUDA(ctx, cudaEventRecord(ctx->edit_ev[0], es));
  GP_CUDA(ctx, gp::launch_edit(p, ctx->sm_count, es, alongside));
  if (!alongside) GP_CUDA(ctx, cudaEventRecord(ctx->edit_ev[1], es));
  ctx->edit_ev_valid = !alongside;
  return GP_OK;
}

// goldpolish-mask / to-upper over the records resident after the edit kernel (or after gp_prep's staging)
static int prep_launch(gp_ctx* ctx, int32_t mode, uint32_t k, int32_t to_upper)
{
  if (ctx->n_contigs == 0 || (!mode && !to_upper)) return GP_OK;
  gp::PrepParams q;
  std::memset(&q, 0, sizeof q);
  q.n_contigs = ctx->n_contigs;
  q.buf[0] = ctx->d_buf0.as<char>();
  q.buf[1] = ctx->d_buf1.as<char>();
  q.cap_off = ctx->d_cap_off.as<uint64_t>();
  q.cur_len = ctx->d_cur_len.as<uint32_t>();
  q.which = ctx->d_which.as<uint8_t>();
  q.dropped = ctx->d_dropped.as<uint8_t>();
  q.k = k; q.mode = mode; q.to_upper = to_upper;
  GP_CUDA(ctx, gp::launch_prep(q, ctx->sm_count, ctx->stream));
  return GP_OK;
}

// edit records: the lengths and buffer indices the edit kernel left, before the mask / to-upper pass moves the records on
// (that pass writes the other buffer, so the kernel's records and origins stay as they are)
static int keep_edit_result(gp_ctx* ctx)
{
  ctx->edits_polish = false;
  ctx->edits_ready = false;
  if (!ctx->cfg.track_edits) return GP_OK;
  const size_t n = std::max<size_t>(ctx->n_contigs, 1);
  GP_CUDA(ctx, ctx->d_elen.ensure(n * 4));
  GP_CUDA(ctx, ctx->d_ewhich.ensure(n));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_elen.p, ctx->d_cur_len.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_ewhich.p, ctx->d_which.p, n, cudaMemcpyDeviceToDevice, ctx->stream));
  ctx->edits_polish = true;
  return GP_OK;
}

// k-mer support: buffers for this polish, counts and bits cleared (stream order: before its first edit kernel).  The
// bitmap of unsupported starts is sized from the draft lengths and the polished records' capacities of this layout (a
// re-run after buffer growth comes through here again); it needs no clearing: a record's words are all written by the
// last count of its contig, and the derivation reads no others.
static int support_begin(gp_ctx* ctx)
{
  ctx->support_polish = false;
  ctx->unsupported_ready = false;
  if (!ctx->cfg.kmer_support) return GP_OK;
  const uint32_t nk = ctx->cfg.nk;
  const size_t n = std::max<size_t>(ctx->n_contigs, 1), nb = std::max<size_t>(ctx->n_batches, 1);
  GP_CUDA(ctx, ctx->d_support.ensure(n * nk * sizeof(gp_kmer_support)));
  GP_CUDA(ctx, ctx->d_sup_steps.ensure(2 * n * 8));
  GP_CUDA(ctx, ctx->d_sup_bits.ensure(nb * nk * 8));
  ctx->sup_draft_words = ctx->h_in_off[ctx->n_contigs] / 32 + ctx->n_contigs;
  ctx->sup_polished_words = ctx->h_cap_off[ctx->n_contigs] / 32 + ctx->n_contigs;
  GP_CUDA(ctx, ctx->d_sup_miss.ensure(std::max<uint64_t>(uint64_t(nk) * (ctx->sup_draft_words + ctx->sup_polished_words), 1) * 4));
  GP_CUDA(ctx, ctx->d_sup_len.ensure(n * 4));
  gp::SupportInput in;
  std::memset(&in, 0, sizeof in);
  in.n = ctx->n_contigs;
  size_t tmp = 0;
  GP_CUDA(ctx, gp::support_count(in, gp::SupportMiss{}, nullptr, nullptr, tmp, ctx->sm_count, ctx->stream));
  GP_CUDA(ctx, ctx->d_sup_tmp.ensure(std::max<size_t>(tmp, 16)));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_support.p, 0, n * nk * sizeof(gp_kmer_support), ctx->stream));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_sup_bits.p, 0, nb * nk * 8, ctx->stream));
  ctx->support_polish = true;
  return GP_OK;
}

// k-mer support of the n contigs ids[0 .. n) (nullptr: all) just polished, and the set bits of the batches whose filters
// are resident for them: batches[0 .. n_batches) (nullptr: 0 .. n_batches - 1)
static int support_launch(gp_ctx* ctx, const uint32_t* ids, uint32_t n, const uint32_t* batches, uint32_t n_batches)
{
  if (!ctx->cfg.kmer_support) return GP_OK;
  const gp_config& c = ctx->cfg;
  gp::SupportInput in;
  std::memset(&in, 0, sizeof in);
  in.n = n;
  in.ids = ids;
  in.draft = ctx->d_input.as<char>();
  in.draft_off = ctx->d_in_off.as<uint64_t>();
  in.buf[0] = ctx->d_buf0.as<char>();
  in.buf[1] = ctx->d_buf1.as<char>();
  in.cap_off = ctx->d_cap_off.as<uint64_t>();
  in.len = ctx->d_cur_len.as<uint32_t>();
  in.which = ctx->d_which.as<uint8_t>();
  in.dropped = ctx->d_dropped.as<uint8_t>();
  in.contig_batch = ctx->d_contig_batch.as<uint32_t>();
  in.bf_pool = ctx->d_bf_pool.as<uint32_t>();
  in.bf_slot = ctx->bf_all_resident ? nullptr : ctx->d_bf_slot.as<uint32_t>();
  in.error = ctx->d_error.as<int>();
  in.counts = ctx->d_support.as<unsigned long long>();
  in.nk = c.nk;
  for (uint32_t i = 0; i < c.nk; i++) in.k[i] = c.k[i];
  const gp::SupportMiss miss{ ctx->d_sup_miss.as<uint32_t>(), ctx->sup_draft_words, ctx->sup_polished_words };
  size_t tmp = ctx->d_sup_tmp.cap;
  GP_CUDA(ctx, gp::support_count(in, miss, ctx->d_sup_steps.as<uint64_t>(), ctx->d_sup_tmp.p, tmp, ctx->sm_count, ctx->stream));
  GP_CUDA(ctx, gp::support_popcount(in.bf_pool, in.bf_slot, batches, 0, n_batches, c.nk, ctx->d_sup_bits.as<unsigned long long>(),
                                    ctx->stream));
  return GP_OK;
}

// the polished lengths the last counts saw, before the mask / to-upper pass changes them
static int support_keep(gp_ctx* ctx)
{
  if (!ctx->cfg.kmer_support || !ctx->n_contigs) return GP_OK;
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_sup_len.p, ctx->d_cur_len.p, size_t(ctx->n_contigs) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  return GP_OK;
}

static int polish_launch(gp_ctx* ctx)
{
  if (int rc = polish_prepare(ctx)) return rc;
  if (int rc = support_begin(ctx)) return rc;
  if (int rc = polish_edit(ctx, ctx->stream, nullptr, 0, nullptr, false)) return rc;
  if (int rc = support_launch(ctx, nullptr, ctx->n_contigs, nullptr, ctx->n_batches)) return rc;
  if (int rc = support_keep(ctx)) return rc;
  if (int rc = keep_edit_result(ctx)) return rc;
  return prep_launch(ctx, ctx->cfg.prep_mode, ctx->cfg.prep_k, ctx->cfg.to_upper);
}

int gp_polish_run(gp_ctx* ctx)
{
  if (!ctx) return GP_ERR_ARG;
  if (!ctx->polish_staged) GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_run before gp_polish_stage");
  if (!ctx->filters_ready)
    GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_run needs the whole filter set resident (build it first; when the filters do not all fit, "
                               "gp_pipeline_run polishes wave by wave)");
  cudaSetDevice(ctx->cfg.device);
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[4], ctx->stream));
  if (int rc = polish_launch(ctx)) return rc;
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[5], ctx->stream));
  ctx->polish_timed = true;
  ctx->stats.polish_launches = ctx->n_contigs ? 2 + ((ctx->cfg.prep_mode || ctx->cfg.to_upper) ? 1 : 0) : 0; // scatter + edit (+ mask) kernels
  ctx->polish_done = true;
  return GP_OK;
}

int gp_prep(gp_ctx* ctx, uint32_t n_records, const char* seqs, const uint64_t* offsets, int32_t mode, uint32_t k,
            int32_t to_upper, char* out_seqs, uint64_t out_cap, uint64_t* out_offsets)
{
  if (!ctx || !offsets || !out_offsets || (!seqs && n_records && offsets[n_records])) return GP_ERR_ARG;
  if (mode < 0 || mode > 2 || (mode && (k == 0 || k > 64))) GP_FAIL(ctx, GP_ERR_ARG, "gp_prep: mode 0..2, k 1..64");
  cudaSetDevice(ctx->cfg.device);
  const uint32_t n = n_records;
  ctx->n_contigs = n;
  ctx->h_len.resize(n);
  ctx->h_in_off.assign(offsets, offsets + n + 1);
  ctx->h_batch.assign(n, 0u);
  for (uint32_t i = 0; i < n; i++) {
    const uint64_t len = offsets[i + 1] - offsets[i];
    if (len >= (1ull << 31)) GP_FAIL(ctx, GP_ERR_ARG, "record longer than 2^31 bases");
    ctx->h_len[i] = uint32_t(len);
  }
  const uint64_t total = offsets[n];
  GP_CUDA(ctx, ctx->d_input.ensure(std::max<uint64_t>(total, 16)));
  GP_CUDA(ctx, ctx->d_in_off.ensure((size_t(n) + 1) * 8));
  GP_CUDA(ctx, ctx->d_cur_len.ensure(std::max<size_t>(n, 1) * 4));
  GP_CUDA(ctx, ctx->d_which.ensure(std::max<size_t>(n, 1)));
  GP_CUDA(ctx, ctx->d_dropped.ensure(std::max<size_t>(n, 1)));
  GP_CUDA(ctx, ctx->d_pnext.ensure(4));
  GP_CUDA(ctx, ctx->d_pcounters.ensure(64));
  GP_CUDA(ctx, ctx->d_error.ensure(4));
  cudaStream_t s = ctx->stream;
  if (total) GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_input.p, seqs, total, cudaMemcpyHostToDevice, s));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_in_off.p, offsets, (size_t(n) + 1) * 8, cudaMemcpyHostToDevice, s));
  ctx->grow = 0;
  if (int rc = polish_layout(ctx)) return rc;
  if (int rc = polish_prepare(ctx)) return rc; // records into buffer 0
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_which.p, 0, std::max<size_t>(n, 1), s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_dropped.p, 0, std::max<size_t>(n, 1), s));
  if (int rc = prep_launch(ctx, mode, k, to_upper)) return rc;
  ctx->polish_staged = false; // the staged contigs (if any) were replaced
  ctx->polish_done = true;
  ctx->edits_polish = false;
  ctx->support_polish = false;
  return gp_polish_fetch(ctx, out_seqs, out_cap, out_offsets, nullptr);
}

int gp_pipeline_run(gp_ctx* ctx)
{
  if (!ctx) return GP_ERR_ARG;
  if (!ctx->build_staged) GP_FAIL(ctx, GP_ERR_STATE, "gp_pipeline_run before gp_build_stage");
  if (!ctx->polish_staged) GP_FAIL(ctx, GP_ERR_STATE, "gp_pipeline_run before gp_polish_stage");
  cudaSetDevice(ctx->cfg.device);
  const gp_config& c = ctx->cfg;
  const uint32_t n = ctx->n_contigs, nb = ctx->n_batches;
  if (ctx->overlap_state == 0 && ctx->pipelined) {
    // first overlapped pass of this context is behind us: did the edit kernel ever see filters arrive while it ran?
    int err = 0;
    GP_CUDA(ctx, cudaMemcpyAsync(&err, ctx->d_error.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->overlap_state == 0) ctx->overlap_state = err == 2 ? -1 : 1; // 2 = its watchdog fired: this device does not co-schedule the kernels
    if (ctx->sm_split_state == 0) sm_split_check(ctx);
  }
  const int algo = ctx->build_algo_resolved;
  const bool overlap = algo == 2 && n && nb && !c.keep_counters && ctx->overlap_state >= 0 && !std::getenv("GP_NO_OVERLAP");
  if (!overlap && ctx->bf_all_resident) { // nothing to overlap with (or the in-order kernel, which fills the SMs): one after the other
    if (int rc = gp_build_run(ctx)) return rc;
    return gp_polish_run(ctx);
  }
  // Launch order of the batches: (overlapped) those with the longest contigs first -- their edit chains are the critical
  // path -- else as given; contigs in the order of their batches, longest first inside a batch.  Waves are runs of
  // wave_batches positions of that order.
  {
    std::vector<uint32_t> maxlen(nb, 0), pos(nb, 0);
    for (uint32_t i = 0; i < n; i++) maxlen[ctx->h_batch[i]] = std::max(maxlen[ctx->h_batch[i]], ctx->h_len[i]);
    ctx->h_batch_order.resize(nb);
    std::iota(ctx->h_batch_order.begin(), ctx->h_batch_order.end(), 0u);
    if (overlap)
      std::stable_sort(ctx->h_batch_order.begin(), ctx->h_batch_order.end(), [&](uint32_t a, uint32_t b) { return maxlen[a] > maxlen[b]; });
    for (uint32_t i = 0; i < nb; i++) pos[ctx->h_batch_order[i]] = i;
    ctx->h_order_pipe.resize(n);
    std::iota(ctx->h_order_pipe.begin(), ctx->h_order_pipe.end(), 0u);
    std::stable_sort(ctx->h_order_pipe.begin(), ctx->h_order_pipe.end(), [&](uint32_t a, uint32_t b) {
      const uint32_t pa = pos[ctx->h_batch[a]], pb = pos[ctx->h_batch[b]];
      return pa != pb ? pa < pb : ctx->h_len[a] > ctx->h_len[b];
    });
    // contigs of every wave: a contiguous range of h_order_pipe
    ctx->h_wave_contig_off.assign(ctx->wave_first.size() + 1, 0);
    for (uint32_t i = 0; i < n; i++) {
      const uint32_t p = pos[ctx->h_batch[i]];
      size_t wv = ctx->wave_batches ? p / ctx->wave_batches : 0;
      if (wv >= ctx->wave_first.size()) wv = ctx->wave_first.size() - 1;
      ctx->h_wave_contig_off[wv + 1]++;
    }
    for (size_t wv = 0; wv < ctx->wave_first.size(); wv++) ctx->h_wave_contig_off[wv + 1] += ctx->h_wave_contig_off[wv];
  }
  cudaStream_t s = ctx->stream;
  GP_CUDA(ctx, ctx->d_batch_order.ensure(std::max<size_t>(nb, 1) * 4));
  GP_CUDA(ctx, ctx->d_batch_done.ensure((size_t(nb) + 1) * 4));
  GP_CUDA(ctx, ctx->d_order_pipe.ensure(std::max<size_t>(n, 1) * 4));
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[2], s));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_batch_order.p, ctx->h_batch_order.data(), size_t(nb) * 4, cudaMemcpyHostToDevice, s));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_order_pipe.p, ctx->h_order_pipe.data(), size_t(n) * 4, cudaMemcpyHostToDevice, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_batch_done.p, 0, (size_t(nb) + 1) * 4, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, gp::kBuildCounters * 8, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.as<unsigned long long>() + 20, 0xFF, 8, s)); // first start time: atomicMin
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_next.p, 0, ctx->wave_first.size() * 4, s));
  const uint64_t per_bf = uint64_t(c.nk) * gp::kBfBytes;
  if (ctx->bf_all_resident) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_bf_pool.p, 0, uint64_t(nb) * per_bf, s));
  if (int rc = upload_bf_slots(ctx, s, true)) return rc;
  if (algo == 2)
    if (int rc = build_stream_tab(ctx, s, true)) return rc;
  if (int rc = polish_prepare(ctx)) return rc;
  if (int rc = support_begin(ctx)) return rc;
  // Per wave: the build kernel signals `launch_dependents` as it starts; the edit kernel (persistent) is launched behind
  // it in the SAME stream with programmatic stream serialization, so it becomes resident while the build runs, takes
  // the wave's contigs in build order and waits for each one's filters.  No event may sit between the two launches;
  // their durations come from device timers.  The next wave's pool clear waits (stream order) for this wave's edit
  // kernel.
  // How the two kernels share the GPU.  Default: the edit kernel gets SMs of its own -- the build launch fills every SM
  // (3 CTAs) and hands E of them back, the edit kernel's whole-SM CTAs land there (and on every SM once the build is
  // through).  E from the work staged: edit ~0.8 us of one warp per draft base and k chain when the warp has a
  // scheduler to itself, build ~9.6 G k-mer ops/s, 12 edit warps per SM at about a third of that speed each (three to
  // a scheduler, L2 busy with the build) -- measured: with less, polishing falls behind the build and the step ends
  // in a tail; every SM given away costs the build a little more than its 1/148.  GP_EDIT_SMS=n fixes E; 0 is the older
  // scheme (every SM: 2 build CTAs + one 3-warp edit CTA), which costs the build more than it looks: an edit warp slows
  // its SM's part of EVERY barrier interval, and the grid barrier waits for the slowest SM.
  uint32_t edit_sms = 0;
  if (overlap) {
    uint64_t draft = 0, steps = 0;
    for (uint32_t i = 0; i < n; i++) draft += ctx->h_len[i];
    for (uint32_t ki = 0; ki < c.nk; ki++) steps += ctx->h_pre[size_t(ki) * (ctx->n_entries + 1) + ctx->n_entries];
    const double edit_s = double(draft) * 0.8e-6, build_s = std::max(1e-6, double(steps) * 32.0 / 9.6e9);
    edit_sms = uint32_t(std::ceil(4.5 * edit_s / build_s / 12.0));
    edit_sms = std::min(std::max(edit_sms, 2u), 24u);
    if (const char* e = std::getenv("GP_EDIT_SMS")) edit_sms = uint32_t(std::max(0, std::atoi(e)));
    if (std::getenv("GP_LEVEL_CTAS") || int(edit_sms) * 2 > ctx->sm_count) edit_sms = 0; // (experiments with other grids)
    if (ctx->sm_split_state < 0) edit_sms = 0; // this device does not deal CTAs to SMs the way the split counts on
  }
  ctx->edit_sms = edit_sms;
  ctx->edit_ctas_per_sm = uint32_t(gp::levels_ctas_per_sm(0));
  ctx->stats.edit_sms = edit_sms;
  int shared_ctas = 2; // build CTAs per SM when the edit kernel shares the SMs
  if (const char* e = std::getenv("GP_EXP_PIPE_CTAS")) shared_ctas = std::max(1, std::atoi(e)); // (experiments)
  uint32_t launches = 0, edit_launches = 0;
  uint32_t* bd = overlap ? ctx->d_batch_done.as<uint32_t>() : nullptr;
  for (size_t wv = 0; wv < ctx->wave_first.size(); wv++) {
    if (!ctx->bf_all_resident) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_bf_pool.p, 0, uint64_t(ctx->wave_count[wv]) * per_bf, s));
    if (algo == 2) { if (int rc = build_launch_levels_wave(ctx, s, wv, bd, overlap && !edit_sms ? shared_ctas : 0, edit_sms)) return rc; }
    else if (int rc = build_launch_inorder_wave(ctx, s, wv)) return rc;
    launches++;
    const uint32_t c0 = ctx->h_wave_contig_off[wv], c1 = ctx->h_wave_contig_off[wv + 1];
    if (c1 > c0) {
      if (wv) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_pnext.p, 0, 4, s));
      if (int rc = polish_edit(ctx, s, ctx->d_order_pipe.as<uint32_t>() + c0, c1 - c0, bd, overlap ? (edit_sms ? 2 : 1) : 0)) return rc;
      edit_launches++;
    }
    // k-mer support of the wave's contigs and filters, before the next wave's pool clear
    if (int rc = support_launch(ctx, ctx->d_order_pipe.as<uint32_t>() + c0, c1 - c0, ctx->d_batch_order.as<uint32_t>() + ctx->wave_first[wv],
                                ctx->wave_count[wv])) return rc;
    if (int rc = wave_payloads_out(ctx, s, wv, algo == 2 && ctx->bf_host_dev)) return rc;
  }
  ctx->bf_streamed = ctx->bf_host_user && ((algo == 2 && ctx->bf_host_dev) || !ctx->bf_all_resident);
  if (int rc = support_keep(ctx)) return rc;
  if (int rc = keep_edit_result(ctx)) return rc;
  if (int rc = prep_launch(ctx, c.prep_mode, c.prep_k, c.to_upper)) return rc;
  GP_CUDA(ctx, cudaEventRecord(ctx->ev[3], s));
  ctx->pipelined = true;
  ctx->build_timed = true;
  ctx->polish_timed = true;
  ctx->stats.build_launches = launches;
  ctx->stats.build_kernel = uint32_t(algo);
  ctx->stats.build_slots = algo == 2 ? ctx->level_slots : 0;
  ctx->stats.level_time_bits = algo == 2 ? ctx->level_time_bits : 0;
  ctx->stats.polish_launches = 1 + edit_launches + ((c.prep_mode || c.to_upper) ? 1 : 0);
  ctx->filters_ready = ctx->bf_all_resident;
  ctx->build_done = true;
  ctx->polish_done = true;
  return GP_OK;
}

// Lengths and dropped flags of the last polish, once it has run without error: a contig that outgrew its buffers, or
// the overlapped edit kernel's watchdog, makes the polish run again here
static int polish_settle(gp_ctx* ctx, std::vector<uint32_t>& len, std::vector<uint8_t>& dropped)
{
  cudaStream_t s = ctx->stream;
  const uint32_t n = ctx->n_contigs;
  len.resize(n);
  dropped.resize(n);
  for (;;) {
    int err = 0;
    GP_CUDA(ctx, cudaMemcpyAsync(&err, ctx->d_error.p, 4, cudaMemcpyDeviceToHost, s));
    if (n) {
      GP_CUDA(ctx, cudaMemcpyAsync(len.data(), ctx->d_cur_len.p, size_t(n) * 4, cudaMemcpyDeviceToHost, s));
      GP_CUDA(ctx, cudaMemcpyAsync(dropped.data(), ctx->d_dropped.p, n, cudaMemcpyDeviceToHost, s));
    }
    GP_CUDA(ctx, cudaStreamSynchronize(s));
    if (!err) break;
    // the polish runs again on the device: from the resident filters, or -- when the pool only ever held one wave --
    // as a whole new pass of the pipeline
    auto rerun = [&]() { ctx->stats.polish_reruns++; return ctx->filters_ready ? polish_launch(ctx) : gp_pipeline_run(ctx); };
    if (err == 2) { // pipelined edit kernel gave up waiting for filters (no co-residency): plain re-run, filters are final now
      ctx->overlap_state = -1; // remembered here: the re-run below clears d_error before gp_pipeline_run could look at it
      if (int rc = rerun()) return rc;
      continue;
    }
    // an edited contig outgrew its buffers: enlarge them and run the polish again
    if (ctx->grow >= 4) GP_FAIL(ctx, GP_ERR_OVERFLOW, "edited contig outgrew its device buffers");
    ctx->grow++;
    if (int rc = polish_layout(ctx)) return rc;
    if (int rc = rerun()) return rc;
  }
  return GP_OK;
}

int gp_polish_fetch(gp_ctx* ctx, char* out_seqs, uint64_t out_cap, uint64_t* out_offsets, uint8_t* out_dropped)
{
  if (!ctx || !out_offsets) return GP_ERR_ARG;
  if (!ctx->polish_done) GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch before gp_polish_run");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t s = ctx->stream;
  const uint32_t n = ctx->n_contigs;
  std::vector<uint32_t> len;
  std::vector<uint8_t> dropped;
  if (int rc = polish_settle(ctx, len, dropped)) return rc;
  uint64_t o = 0;
  for (uint32_t i = 0; i < n; i++) {
    out_offsets[i] = o;
    if (!dropped[i]) o += len[i];
    if (out_dropped) out_dropped[i] = dropped[i];
  }
  out_offsets[n] = o;
  if (o > out_cap || (o && !out_seqs)) GP_FAIL(ctx, GP_ERR_ARG, "output buffer too small (needed size is in out_offsets[n])");
  if (o) {
    GP_CUDA(ctx, ctx->d_out.ensure(o));
    GP_CUDA(ctx, ctx->d_out_off.ensure((size_t(n) + 1) * 8));
    GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_out_off.p, out_offsets, (size_t(n) + 1) * 8, cudaMemcpyHostToDevice, s));
    const uint32_t grid = std::min<uint32_t>(n, uint32_t(ctx->sm_count) * 8u);
    gather_contigs_kernel<<<grid, 256, 0, s>>>(ctx->d_buf0.as<char>(), ctx->d_buf1.as<char>(), ctx->d_cap_off.as<uint64_t>(),
                                               ctx->d_which.as<uint8_t>(), ctx->d_out_off.as<uint64_t>(), ctx->d_out.as<char>(), n);
    GP_CUDA(ctx, cudaGetLastError());
    GP_CUDA(ctx, cudaMemcpyAsync(out_seqs, ctx->d_out.p, o, cudaMemcpyDeviceToHost, s));
    GP_CUDA(ctx, cudaStreamSynchronize(s));
  }
  return GP_OK;
}

int gp_polish(gp_ctx* ctx, uint32_t n_contigs, const char* seqs, const uint64_t* offsets, const uint32_t* contig_batch,
              char* out_seqs, uint64_t out_cap, uint64_t* out_offsets, uint8_t* out_dropped)
{
  int rc = gp_polish_stage(ctx, n_contigs, seqs, offsets, contig_batch);
  if (rc) return rc;
  if ((rc = gp_polish_run(ctx))) return rc;
  return gp_polish_fetch(ctx, out_seqs, out_cap, out_offsets, out_dropped);
}

// ------------------------------------------------------------------------------------
// edit records (derived from the polished records and the origin map, gp_edits.cu)
// ------------------------------------------------------------------------------------
static int derive_edits(gp_ctx* ctx, const std::vector<uint8_t>& dropped)
{
  cudaStream_t s = ctx->stream;
  const uint32_t n = ctx->n_contigs;
  std::vector<uint32_t> elen(n);
  if (n) GP_CUDA(ctx, cudaMemcpyAsync(elen.data(), ctx->d_elen.p, size_t(n) * 4, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  std::vector<uint64_t> bnd(size_t(n) + 1, 0);
  for (uint32_t c = 0; c < n; c++) bnd[c + 1] = bnd[c] + (dropped[c] ? 0 : uint64_t(elen[c]) + 1);
  const uint64_t n_bnd = bnd[n];
  GP_CUDA(ctx, ctx->d_bnd_off.ensure((size_t(n) + 1) * 8));
  GP_CUDA(ctx, ctx->d_eflags.ensure((n_bnd + 1) * 8));
  GP_CUDA(ctx, ctx->d_edit_coff.ensure((size_t(n) + 1) * 8));
  GP_CUDA(ctx, ctx->d_edit_err.ensure(4));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bnd_off.p, bnd.data(), (size_t(n) + 1) * 8, cudaMemcpyHostToDevice, s));
  GP_CUDA(ctx, cudaMemsetAsync(ctx->d_edit_err.p, 0x7F, 4, s)); // atomicMin target
  gp::EditsInput in;
  in.n_contigs = n;
  in.draft = ctx->d_input.as<char>();
  in.draft_off = ctx->d_in_off.as<uint64_t>();
  in.buf[0] = ctx->d_buf0.as<char>();
  in.buf[1] = ctx->d_buf1.as<char>();
  in.orig[0] = ctx->d_orig0.as<uint32_t>();
  in.orig[1] = ctx->d_orig1.as<uint32_t>();
  in.cap_off = ctx->d_cap_off.as<uint64_t>();
  in.len = ctx->d_elen.as<uint32_t>();
  in.which = ctx->d_ewhich.as<uint8_t>();
  in.bnd_off = ctx->d_bnd_off.as<uint64_t>();
  in.error = ctx->d_edit_err.as<int>();
  uint64_t* flags = ctx->d_eflags.as<uint64_t>();
  size_t tmp = 0;
  GP_CUDA(ctx, gp::edits_count(in, n_bnd, flags, nullptr, tmp, s));
  GP_CUDA(ctx, ctx->d_etmp.ensure(std::max<size_t>(tmp, 16)));
  tmp = ctx->d_etmp.cap;
  GP_CUDA(ctx, gp::edits_count(in, n_bnd, flags, ctx->d_etmp.p, tmp, s));
  uint64_t total = 0;
  int bad = 0;
  GP_CUDA(ctx, cudaMemcpyAsync(&total, flags + n_bnd, 8, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaMemcpyAsync(&bad, ctx->d_edit_err.p, 4, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  if (bad != 0x7F7F7F7F)
    GP_FAIL(ctx, GP_ERR_STATE, "edit records: the origins of contig " + std::to_string(bad - 1) +
                               " do not increase strictly along the polished record; no records are derived");
  const uint32_t n_rec = uint32_t(total);
  if ((total >> 32) != n_rec) GP_FAIL(ctx, GP_ERR_STATE, "edit records: record starts and ends do not pair up");
  GP_CUDA(ctx, ctx->d_rec_c.ensure(std::max<size_t>(n_rec, 1) * 4));
  GP_CUDA(ctx, ctx->d_rec_i.ensure(std::max<size_t>(n_rec, 1) * 4));
  GP_CUDA(ctx, ctx->d_rec_j.ensure(std::max<size_t>(n_rec, 1) * 4));
  GP_CUDA(ctx, ctx->d_edits.ensure(std::max<size_t>(n_rec, 1) * sizeof(gp_edit)));
  GP_CUDA(ctx, ctx->d_alen.ensure((size_t(n_rec) + 1) * 8));
  tmp = 0;
  GP_CUDA(ctx, gp::edits_fill(in, n_bnd, flags, n_rec, nullptr, nullptr, nullptr, nullptr, ctx->d_alen.as<uint64_t>(), nullptr,
                              nullptr, tmp, s));
  GP_CUDA(ctx, ctx->d_etmp.ensure(std::max<size_t>(tmp, 16)));
  tmp = ctx->d_etmp.cap;
  GP_CUDA(ctx, gp::edits_fill(in, n_bnd, flags, n_rec, ctx->d_rec_c.as<uint32_t>(), ctx->d_rec_i.as<uint32_t>(),
                              ctx->d_rec_j.as<uint32_t>(), ctx->d_edits.as<gp_edit>(), ctx->d_alen.as<uint64_t>(),
                              ctx->d_edit_coff.as<uint64_t>(), ctx->d_etmp.p, tmp, s));
  uint64_t bytes = 0;
  GP_CUDA(ctx, cudaMemcpyAsync(&bytes, ctx->d_alen.as<uint64_t>() + n_rec, 8, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  GP_CUDA(ctx, ctx->d_alleles.ensure(std::max<uint64_t>(bytes, 16)));
  GP_CUDA(ctx, gp::edits_alleles(in, n_rec, ctx->d_rec_c.as<uint32_t>(), ctx->d_rec_i.as<uint32_t>(), ctx->d_rec_j.as<uint32_t>(),
                                 ctx->d_alen.as<uint64_t>(), ctx->d_edits.as<gp_edit>(), ctx->d_alleles.as<char>(), s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  ctx->n_edits = n_rec;
  ctx->n_allele_bytes = bytes;
  ctx->edits_ready = true;
  return GP_OK;
}

int gp_polish_fetch_edits(gp_ctx* ctx, uint64_t* contig_edit_off, gp_edit* edits, uint64_t edits_cap, char* alleles,
                          uint64_t alleles_cap, uint64_t needed[2])
{
  if (!ctx || !contig_edit_off || !needed) return GP_ERR_ARG;
  if (!ctx->cfg.track_edits) GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch_edits needs gp_config.track_edits = 1");
  if (!ctx->polish_done || !ctx->edits_polish)
    GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch_edits before gp_polish_run / gp_pipeline_run");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t s = ctx->stream;
  std::vector<uint32_t> len;
  std::vector<uint8_t> dropped;
  if (int rc = polish_settle(ctx, len, dropped)) return rc;
  if (!ctx->edits_ready)
    if (int rc = derive_edits(ctx, dropped)) return rc;
  const uint32_t n = ctx->n_contigs;
  needed[0] = ctx->n_edits;
  needed[1] = ctx->n_allele_bytes;
  GP_CUDA(ctx, cudaMemcpyAsync(contig_edit_off, ctx->d_edit_coff.p, (size_t(n) + 1) * 8, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  if (edits_cap < ctx->n_edits || alleles_cap < ctx->n_allele_bytes || (ctx->n_edits && !edits) ||
      (ctx->n_allele_bytes && !alleles))
    GP_FAIL(ctx, GP_ERR_ARG, "edit record buffers too small (needed[0] records, needed[1] allele bytes)");
  if (ctx->n_edits)
    GP_CUDA(ctx, cudaMemcpyAsync(edits, ctx->d_edits.p, ctx->n_edits * sizeof(gp_edit), cudaMemcpyDeviceToHost, s));
  if (ctx->n_allele_bytes)
    GP_CUDA(ctx, cudaMemcpyAsync(alleles, ctx->d_alleles.p, ctx->n_allele_bytes, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  return GP_OK;
}

int gp_polish_fetch_support(gp_ctx* ctx, gp_kmer_support* out, uint64_t* filter_bits_set)
{
  if (!ctx) return GP_ERR_ARG;
  if (!ctx->cfg.kmer_support) GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch_support needs gp_config.kmer_support = 1");
  if (!ctx->polish_done || !ctx->support_polish)
    GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch_support before gp_polish_run / gp_pipeline_run");
  if (!out && ctx->n_contigs) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t s = ctx->stream;
  std::vector<uint32_t> len;
  std::vector<uint8_t> dropped;
  if (int rc = polish_settle(ctx, len, dropped)) return rc;
  const uint32_t nk = ctx->cfg.nk;
  if (ctx->n_contigs)
    GP_CUDA(ctx, cudaMemcpyAsync(out, ctx->d_support.p, size_t(ctx->n_contigs) * nk * sizeof(gp_kmer_support), cudaMemcpyDeviceToHost, s));
  if (filter_bits_set && ctx->n_batches)
    GP_CUDA(ctx, cudaMemcpyAsync(filter_bits_set, ctx->d_sup_bits.p, size_t(ctx->n_batches) * nk * 8, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  return GP_OK;
}

// runs of unsupported k-mers (gp_support.cu): segments (contig, record, k) of the bitmap as one flat range of words,
// counted, scanned and filled on the device
static int derive_unsupported(gp_ctx* ctx, const std::vector<uint8_t>& dropped)
{
  cudaStream_t s = ctx->stream;
  const uint32_t n = ctx->n_contigs, nk = ctx->cfg.nk, n_seg = n * 2 * nk;
  std::vector<uint32_t> plen(n);
  if (n) GP_CUDA(ctx, cudaMemcpyAsync(plen.data(), ctx->d_sup_len.p, size_t(n) * 4, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  std::vector<uint64_t> seg(size_t(n_seg) + 1, 0);
  for (uint32_t c = 0; c < n; c++)
    for (uint32_t r = 0; r < 2; r++) {
      // lengths as support_count_kernel reads the records
      const uint64_t len = r ? (dropped[c] ? 0 : std::min<uint64_t>(plen[c], ctx->h_cap_off[c + 1] - ctx->h_cap_off[c]))
                             : ctx->h_in_off[c + 1] - ctx->h_in_off[c];
      for (uint32_t j = 0; j < nk; j++) {
        const size_t i = (size_t(c) * 2 + r) * nk + j;
        seg[i + 1] = seg[i] + (len >= ctx->cfg.k[j] ? (len + 31) / 32 : 0);
      }
    }
  const uint64_t n_words = seg[n_seg];
  GP_CUDA(ctx, ctx->d_uns_seg.ensure((size_t(n_seg) + 1) * 8));
  GP_CUDA(ctx, ctx->d_uns_off.ensure((size_t(n_seg) + 1) * 8));
  GP_CUDA(ctx, ctx->d_uns_runcnt.ensure(std::max<uint64_t>(n_words, 1) * 8));
  GP_CUDA(ctx, ctx->d_uns_misscnt.ensure(std::max<uint64_t>(n_words, 1) * 4));
  GP_CUDA(ctx, cudaMemcpyAsync(ctx->d_uns_seg.p, seg.data(), (size_t(n_seg) + 1) * 8, cudaMemcpyHostToDevice, s));
  gp::UnsupportedInput in;
  std::memset(&in, 0, sizeof in);
  in.miss = ctx->d_sup_miss.as<uint32_t>();
  in.draft_words = ctx->sup_draft_words;
  in.polished_words = ctx->sup_polished_words;
  in.draft_off = ctx->d_in_off.as<uint64_t>();
  in.cap_off = ctx->d_cap_off.as<uint64_t>();
  in.seg_off = ctx->d_uns_seg.as<uint64_t>();
  in.n_seg = n_seg;
  in.nk = nk;
  for (uint32_t j = 0; j < nk; j++) in.k[j] = ctx->cfg.k[j];
  uint64_t* run_cnt = ctx->d_uns_runcnt.as<uint64_t>();
  uint32_t* miss_cnt = ctx->d_uns_misscnt.as<uint32_t>();
  size_t tmp = 0;
  GP_CUDA(ctx, gp::unsupported_count(in, n_words, run_cnt, miss_cnt, nullptr, tmp, s));
  GP_CUDA(ctx, ctx->d_uns_tmp.ensure(std::max<size_t>(tmp, 16)));
  tmp = ctx->d_uns_tmp.cap;
  GP_CUDA(ctx, gp::unsupported_count(in, n_words, run_cnt, miss_cnt, ctx->d_uns_tmp.p, tmp, s));
  uint64_t total = 0;
  if (n_words) GP_CUDA(ctx, cudaMemcpyAsync(&total, run_cnt + n_words - 1, 8, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  GP_CUDA(ctx, ctx->d_uns_runs.ensure(std::max<uint64_t>(total, 1) * sizeof(gp_unsupported_run)));
  if (total) GP_CUDA(ctx, cudaMemsetAsync(ctx->d_uns_runs.p, 0, total * sizeof(gp_unsupported_run), s));
  GP_CUDA(ctx, gp::unsupported_fill(in, n_words, run_cnt, miss_cnt, ctx->d_uns_runs.as<gp_unsupported_run>(), ctx->d_uns_off.as<uint64_t>(), s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  ctx->n_unsupported = total;
  ctx->unsupported_ready = true;
  return GP_OK;
}

int gp_polish_fetch_unsupported(gp_ctx* ctx, uint64_t* run_off, gp_unsupported_run* runs, uint64_t cap, uint64_t* needed)
{
  if (!ctx || !run_off || !needed) return GP_ERR_ARG;
  if (!ctx->cfg.kmer_support) GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch_unsupported needs gp_config.kmer_support = 1");
  if (!ctx->polish_done || !ctx->support_polish)
    GP_FAIL(ctx, GP_ERR_STATE, "gp_polish_fetch_unsupported before gp_polish_run / gp_pipeline_run");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t s = ctx->stream;
  std::vector<uint32_t> len;
  std::vector<uint8_t> dropped;
  if (int rc = polish_settle(ctx, len, dropped)) return rc;
  if (!ctx->unsupported_ready)
    if (int rc = derive_unsupported(ctx, dropped)) return rc;
  const size_t n_off = size_t(ctx->n_contigs) * 2 * ctx->cfg.nk + 1;
  *needed = ctx->n_unsupported;
  GP_CUDA(ctx, cudaMemcpyAsync(run_off, ctx->d_uns_off.p, n_off * 8, cudaMemcpyDeviceToHost, s));
  GP_CUDA(ctx, cudaStreamSynchronize(s));
  if (cap < ctx->n_unsupported || (ctx->n_unsupported && !runs))
    GP_FAIL(ctx, GP_ERR_ARG, "run buffer too small (needed: *needed runs)");
  if (ctx->n_unsupported) {
    GP_CUDA(ctx, cudaMemcpyAsync(runs, ctx->d_uns_runs.p, ctx->n_unsupported * sizeof(gp_unsupported_run), cudaMemcpyDeviceToHost, s));
    GP_CUDA(ctx, cudaStreamSynchronize(s));
  }
  return GP_OK;
}

// ------------------------------------------------------------------------------------
// flagged regions (derived from the soft-masking of ntedit.cpp:1131-1146)
// ------------------------------------------------------------------------------------
uint64_t gp_flagged_bed(const char* seqs, const uint64_t* offsets, uint32_t n_records, uint32_t* run_record,
                        uint64_t* run_start, uint64_t* run_end, uint64_t cap)
{
  if (!offsets || (!seqs && n_records && offsets[n_records])) return 0;
  uint64_t n = 0;
  for (uint32_t r = 0; r < n_records; r++) {
    const char* s = seqs + offsets[r];
    const uint64_t len = offsets[r + 1] - offsets[r];
    for (uint64_t i = 0; i < len;) {
      if (s[i] < 'a' || s[i] > 'z') { i++; continue; }
      uint64_t j = i + 1;
      while (j < len && s[j] >= 'a' && s[j] <= 'z') j++;
      if (n < cap) {
        if (run_record) run_record[n] = r;
        if (run_start) run_start[n] = i;
        if (run_end) run_end[n] = j;
      }
      n++;
      i = j;
    }
  }
  return n;
}

// ------------------------------------------------------------------------------------
// host-side rules
// ------------------------------------------------------------------------------------
int gp_kmer_threshold(uint64_t mappings_bases)
{ // src/goldpolish_targeted_bfs.cpp:45-53
  const double a = 4.66943, b = 2.11391e-07;
  const int t = int(std::round(a + double(mappings_bases) * b));
  return std::min(t, 13);
}

uint64_t gp_mappings_cap(uint64_t target_len, double subsample_max_per_10kbp)
{ // src/goldpolish_targeted_bfs.cpp:96-99
  return uint64_t(double(target_len) * subsample_max_per_10kbp / 10000.0);
}

int gp_guard_rejects(uint64_t input_bytes, uint64_t output_bytes)
{ // scripts/goldpolish-ntedit:31-34: bc scale=4 truncates the quotient, then "< 0.75"
  if (input_bytes == 0) return 0;
  return (output_bytes * 10000ull) / input_bytes < 7500ull ? 1 : 0;
}

// ------------------------------------------------------------------------------------
// roof microbenchmark
// ------------------------------------------------------------------------------------
int gp_roof_microbench(gp_ctx* ctx, uint32_t warps, uint32_t iters, uint64_t region_bytes, double* sectors_per_s, float* ms)
{
  if (!ctx || !sectors_per_s || warps == 0 || iters == 0 || region_bytes < 4096) return GP_ERR_ARG;
  cudaSetDevice(ctx->cfg.device);
  DevBuf cbf, bf;
  GP_CUDA(ctx, cbf.ensure(std::max<uint64_t>(uint64_t(warps) * region_bytes, gp::kCbfCounters * 4)));
  cudaError_t e = bf.ensure(uint64_t(warps) * gp::kBfBytes);
  if (e != cudaSuccess) { cbf.release(); GP_CUDA(ctx, e); }
  cudaStream_t s = ctx->stream;
  // same L2 conditions as the kernels the roofs are for: the HBM shape (mode 0..2) runs with the whole L2 as normal
  // cache; the L2 shapes (mode 3..5, one shared 40 MiB array) get the persisting window the level kernel uses
  int mode = 0;
  if (const char* m = std::getenv("GP_ROOF_MODE")) mode = std::atoi(m);
  {
    cudaStreamSynchronize(s);
    const bool want = mode >= 3 && ctx->l2_persist_max > 0 && !(std::getenv("GP_L2_PERSIST") && std::getenv("GP_L2_PERSIST")[0] == '0');
    cudaStreamAttrValue av;
    std::memset(&av, 0, sizeof av);
    if (want) {
      av.accessPolicyWindow.base_ptr = cbf.p;
      av.accessPolicyWindow.num_bytes = gp::kCbfCounters * 4;
      av.accessPolicyWindow.hitRatio = 1.0f;
      av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want ? size_t(ctx->l2_persist_max) : 0) != cudaSuccess) cudaGetLastError();
    cudaCtxResetPersistingL2Cache();
    cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &av);
    ctx->l2_window_set = false; // the next build claims its own window again
    ctx->l2_roof_window = want;
  }
  cudaMemsetAsync(cbf.p, 0, uint64_t(warps) * region_bytes, s);
  cudaMemsetAsync(bf.p, 0, uint64_t(warps) * gp::kBfBytes, s);
  cudaEvent_t a, b;
  cudaEventCreate(&a); cudaEventCreate(&b);
  gp::launch_roof(cbf.as<uint8_t>(), bf.as<uint32_t>(), region_bytes, std::min(iters, 64u), warps, s); // warm-up
  cudaEventRecord(a, s);
  gp::launch_roof(cbf.as<uint8_t>(), bf.as<uint32_t>(), region_bytes, iters, warps, s);
  cudaEventRecord(b, s);
  e = cudaStreamSynchronize(s);
  float t = 0;
  cudaEventElapsedTime(&t, a, b);
  cudaEventDestroy(a); cudaEventDestroy(b);
  if (ctx->l2_roof_window) { // leave no window / set-aside behind
    cudaStreamAttrValue av;
    std::memset(&av, 0, sizeof av);
    cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &av);
    cudaCtxResetPersistingL2Cache();
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0);
    ctx->l2_roof_window = false;
  }
  cbf.release(); bf.release();
  GP_CUDA(ctx, e);
  if (ms) *ms = t;
  // modes 3..5 touch 4 sectors per iteration (one round), the build-kernel mix 8
  const int touches = mode >= 3 ? 4 : 8;
  *sectors_per_s = double(warps) * iters * 32.0 * touches / (double(t) * 1e-3);
  return GP_OK;
}

} // extern "C"
