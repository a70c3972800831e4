// ntEdit scan / edit loop on the GPU (sm_100a): one warp per contig, all k rounds chained.
//
// Replaces kmerizeAndCorrect and its helpers (bcgsc/goldpolish subprojects/ntedit/ntedit.cpp
// :1414-1771, :392-413, :441-451, :480-777, :939-1411) plus the FASTA body of writeEditsToFile
// (:797-935) and the k-chain of scripts/goldpolish-ntedit:20-29.
//
// The contig is a sequential state machine (every edit changes what the next position sees),
// so parallelism lives *inside* a decision:
//   * scan: 32 consecutive k-mer windows are hashed and looked up at once; the first absent
//     window / non-IUPAC base / end of contig is found with a ballot;
//   * look-ahead and substitution checks: lane j holds window j, the every-3rd sample set is
//     a lane mask, the counts are ballot + popc;
//   * insertion / deletion search: the 341 insertion strings and <=10 deletions are spread
//     over the lanes, each lane rolling its own candidate; the winner (support, then the
//     reference's evaluation order for ties) is a warp max-reduction.
// The reference's rope (vector<seqNode>) is kept literally in global memory and mutated by
// lane 0 with the reference's own slot arithmetic, because its low-complexity rollback
// (:1038-1100) leaves holes whose position decides what the writer emits.  Hashing never walks
// the rope: the window and the characters ahead of the tail cursor live in a shared-memory
// stream ring refilled from the rope, window hashes come 32 at a time from XOR scans, and the
// presence bits of the next 64 windows are cached so that a run of soft-masked positions costs
// one filter lookup phase per position.
#include "gp_common.cuh"
#include "gp_kernels.cuh"

#include <cstdlib>

namespace gp {

constexpr int kEditWarps = 4;
constexpr uint32_t kFull = 0xffffffffu;

struct Cur {
  uint32_t pos, idx; // (seq_i, node_index) of the reference
  EdNode n;          // cached nodes[idx]; type -2 when idx is past the vector
};

constexpr uint32_t kVBuf = 256; // stream ring (power of two)

struct WS {
  char* seq;
  uint32_t len;
  EdNode* nd;
  uint32_t nn, ncap;
  const uint32_t* bf;
  uint32_t k, jump, icap;
  uint64_t mul1, mul2, mul3;
  float thrM, thrE, thrD;
  uint32_t max_ins, max_del;
  int mode, mask;
  Cur h, t, m;
  HashState hs;      // hash of the current window (valid inside the trigger handler)
  // the stream around the window: vb[i & 255] = character with absolute stream index i;
  // [hp, hp+k) is the window, [hp+k, ve) the characters ahead of the tail cursor
  unsigned char* vb;
  unsigned char* kmer;       // 32 bytes: the window a re-seed starts from (make_edit)
  // candidate-search tables (shared memory): per-round seed tables and per-call staging
  const unsigned char* code; // byte -> 0 none, 1 A, 2 C, 3 G, 4 T (either case)
  uint64_t* seedt;           // [0..4] F, [8..12] F rotated by k, [16..23] R (by c & 7), [24..31] R rotated by k
  uint64_t* stage;           // [0..31] outF, [32..63] outR, [64..127] inF, [128..191] inRk
  uint64_t* com;             // per call: common chains of the insertion search, [0..159] forward (length L-1, roll kk), [160..319] reverse
  const uint64_t* insF;      // per round: [(j * 3 + d - 1) * 32 + kk] = term of inserted base d (C, G, T) that entered at roll j,
  const uint64_t* insR;      //            seen at roll kk (0 while kk < j), forward / reverse strand
  uint32_t hp, ve;
  bool exhausted;    // refilling hit the end of the stream
  // two blocks of 32 windows starting at absolute index B (lane j: windows B+j and B+32+j)
  bool blk_valid;
  uint32_t B;
  uint64_t f0, r0, f1, r1;
  uint64_t pres;     // bit i: window B+i is in the filter
  uint64_t acc;      // bit i: character B+k+i exists and is an accepted base
  uint64_t exist;    // bit i: character B+k+i exists
  uint64_t samp;     // bit kk: kk % jump == 0 && kk < k
  int err;
  uint32_t lane;
  uint32_t n_trig, n_edit, n_mask, n_roll;
};

// seeds through the per-round shared tables instead of the switch statements of gp_common.cuh (branchy on a
// latency-bound warp) and instead of rotating by a runtime k (two modulo operations per srol)
__device__ __forceinline__ uint64_t sF(const WS& w, uint32_t c) { return w.seedt[w.code[c & 255u]]; }       // seedTab[c]
__device__ __forceinline__ uint64_t sFk(const WS& w, uint32_t c) { return w.seedt[8 + w.code[c & 255u]]; }  // ... rotated by k
__device__ __forceinline__ uint64_t sR(const WS& w, uint32_t c) { return w.seedt[16 + (c & 7u)]; }          // seedTab[c & cpOff]
__device__ __forceinline__ uint64_t sRk(const WS& w, uint32_t c) { return w.seedt[24 + (c & 7u)]; }         // ... rotated by k
// rolling update (nthash.hpp:122-131, 143-152) and last-base replacement (:134-140, 154-169)
__device__ __forceinline__ void ws_roll(const WS& w, HashState& h, uint32_t out, uint32_t in)
{
  h.fh = srol1(h.fh) ^ sF(w, in) ^ sFk(w, out);
  h.rh = sror1(h.rh ^ sRk(w, in) ^ sR(w, out));
}
__device__ __forceinline__ void ws_changelast(const WS& w, HashState& h, uint32_t out, uint32_t in)
{
  h.fh ^= sF(w, out) ^ sF(w, in);
  h.rh = sror1(srol1(h.rh) ^ sRk(w, out) ^ sRk(w, in));
}

__device__ __forceinline__ bool is_accepted(uint32_t c)
{ // isAcceptedBase(toupper(c)), ntedit.cpp:363-367
  c &= ~0x20u; // toupper for letters; non-letters never match below either way
  return c == 'A' || c == 'T' || c == 'G' || c == 'C' || c == 'R' || c == 'Y' || c == 'S' || c == 'W' ||
         c == 'K' || c == 'M' || c == 'B' || c == 'D' || c == 'H' || c == 'V';
}
__device__ __forceinline__ uint32_t to_upper(uint32_t c) { return (c >= 'a' && c <= 'z') ? c - 32u : c; }
__device__ __forceinline__ uint32_t to_lower(uint32_t c) { return (c >= 'A' && c <= 'Z') ? c + 32u : c; }
__device__ __forceinline__ unsigned char rc_char(uint32_t c)
{ // RC, ntedit.cpp:369-388
  switch (c) {
  case 'A': case 'a': return 'T';
  case 'T': case 't': return 'A';
  case 'G': case 'g': return 'C';
  case 'C': case 'c': return 'G';
  default: return 'N';
  }
}

__device__ __forceinline__ EdNode ld_node(const EdNode* p)
{
  const int4 v = *reinterpret_cast<const int4*>(p);
  EdNode n;
  n.type = v.x; n.s = uint32_t(v.y); n.e = uint32_t(v.z); n.c = uint32_t(v.w);
  return n;
}
__device__ __forceinline__ void st_node(EdNode* p, const EdNode& n)
{
  *reinterpret_cast<int4*>(p) = make_int4(n.type, int(n.s), int(n.e), int(n.c));
}

// rotate both halves right by s (inverse of srol)
__device__ __forceinline__ uint64_t sror(uint64_t v, uint32_t s)
{
  const uint32_t a = s % 31u, b = s % 33u;
  uint64_t hi = v >> 33, lo = v & 0x1FFFFFFFFULL;
  hi = ((hi >> a) | (hi << (31u - a))) & 0x7FFFFFFFULL;
  lo = ((lo >> b) | (lo << (33u - b))) & 0x1FFFFFFFFULL;
  return (hi << 33) | lo;
}

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p)
{
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// A filter word.  The build kernel may be writing OTHER batches' filters into the same pool while this kernel runs, so
// the non-coherent path (ld.global.nc / __ldg) is out: it is only defined for data that nobody writes during the
// kernel's lifetime.  ld.global.cg reads L2, where the build kernel's `red.or` land.  (An ordinary L1-cached load after
// the ld.acquire.gpu of the batch's flag would also be legal; measured, it changes nothing: 237 vs 233 ms for the
// slowest contig of the config-3 data set, 47.8 vs 45 ms for config 2 -- the chain is instruction latency, not lookups.)
__device__ __forceinline__ uint32_t ld_filter(const uint32_t* p)
{
#ifdef GP_EDIT_FILTER_LOAD_CA
  return __ldca(p);
#else
  return __ldcg(p);
#endif
}

__device__ __forceinline__ bool bf_contains(const WS& w, uint64_t fh, uint64_t rh)
{ // btllib KmerBloomFilter::contains with the four ntHash values (ntedit.cpp:1470)
  const uint64_t b = fh + rh;
  uint64_t h1 = b * w.mul1, h2 = b * w.mul2, h3 = b * w.mul3;
  h1 ^= h1 >> kMultiShift; h2 ^= h2 >> kMultiShift; h3 ^= h3 >> kMultiShift;
  const uint32_t n0 = bf_index(b), n1 = bf_index(h1), n2 = bf_index(h2), n3 = bf_index(h3);
  const uint32_t w0 = ld_filter(w.bf + (n0 >> 5)), w1 = ld_filter(w.bf + (n1 >> 5));
  const uint32_t w2 = ld_filter(w.bf + (n2 >> 5)), w3 = ld_filter(w.bf + (n3 >> 5));
  return ((w0 >> (n0 & 31u)) & (w1 >> (n1 & 31u)) & (w2 >> (n2 & 31u)) & (w3 >> (n3 & 31u)) & 1u) != 0u;
}
__device__ __forceinline__ bool bf_contains(const WS& w, const HashState& h) { return bf_contains(w, h.fh, h.rh); }

// ---- rope cursors (getCharacter :667-678, increment :681-699) -------------------------
__device__ __forceinline__ void cur_load(const WS& w, Cur& c)
{
  if (c.idx < w.nn) c.n = ld_node(w.nd + c.idx);
  else c.n.type = -2;
}
__device__ __forceinline__ uint32_t cur_char(const WS& w, const Cur& c)
{
  if (c.n.type == 0) return c.pos < w.len ? (unsigned char)w.seq[c.pos] : 0u;
  if (c.n.type == 1) return c.n.c;
  return 0u;
}
__device__ __forceinline__ void cur_increment(const WS& w, Cur& c)
{
  if (c.n.type == 0) {
    c.pos++;
    if (c.pos > c.n.e) {
      c.idx++;
      cur_load(w, c);
      if (c.n.type == 0) c.pos = c.n.s;
    }
  } else if (c.n.type == 1) {
    c.idx++;
    cur_load(w, c);
    if (c.n.type == 0) c.pos = c.n.s;
  }
}
// `steps` increments; inside a draft range they collapse to one addition
__device__ __forceinline__ void cur_advance(const WS& w, Cur& c, uint32_t steps)
{
  while (steps) {
    if (c.n.type == 0 && c.pos < c.n.e) {
      const uint32_t d = min(steps, c.n.e - c.pos);
      c.pos += d;
      steps -= d;
    } else {
      cur_increment(w, c);
      steps--;
    }
  }
}
__device__ __forceinline__ bool cur_dead(const WS& w, const Cur& c) { return c.pos >= w.len || c.idx >= w.nn; }

__device__ __forceinline__ uint32_t v_at(const WS& w, uint32_t abs_i) { return w.vb[abs_i & (kVBuf - 1)]; }
__device__ __forceinline__ uint32_t ring_at(const WS& w, uint32_t j) { return v_at(w, w.hp + j); }
__device__ __forceinline__ uint32_t ahead_at(const WS& w, uint32_t j) { return v_at(w, w.hp + w.k + j); }
__device__ __forceinline__ uint32_t ahead_count(const WS& w) { return w.ve - (w.hp + w.k); }

// Extend the stream buffer to absolute index `upto` by walking the rope from the
// materialisation cursor exactly as successive roll() calls would move the tail cursor (:958-966).
__device__ __forceinline__ void stream_fill(WS& w, uint32_t upto)
{
  if (w.ve >= upto || w.exhausted) return;
  while (w.ve < upto && !w.exhausted) {
    if (cur_dead(w, w.m)) { w.exhausted = true; break; }
    if (w.m.n.type == 0 && w.m.pos < w.m.n.e && w.m.pos + 1 < w.len) {
      const uint32_t run = min(min(w.m.n.e, w.len - 1) - w.m.pos, min(upto - w.ve, 32u));
      if (w.lane < run) w.vb[(w.ve + w.lane) & (kVBuf - 1)] = (unsigned char)w.seq[w.m.pos + 1 + w.lane];
      w.m.pos += run;
      w.ve += run;
      continue;
    }
    cur_increment(w, w.m);
    if (cur_dead(w, w.m)) { w.exhausted = true; break; }
    if (w.lane == 0) w.vb[w.ve & (kVBuf - 1)] = (unsigned char)cur_char(w, w.m);
    w.ve++;
  }
  __syncwarp();
}

__device__ __forceinline__ uint64_t xor_scan_incl(uint64_t v, uint32_t lane)
{
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint64_t u = __shfl_up_sync(kFull, v, o);
    if (lane >= (uint32_t)o) v ^= u;
  }
  return v;
}

// Hash and look up the 32 windows that start at absolute indices Bp .. Bp+31 (lane j: window
// Bp+j).  ntHash is XOR-linear in the per-base seeds: with U_i = srol^(62-i)(seed(c_i)) and
// W_i = srol^i(cseed(c_i)) over the 63 characters c_i = stream[Bp+i], a window's forward hash
// is sror^(63-j-k) of the XOR of U over its k characters and its reverse hash sror^j of the
// XOR of W, so two 64-element XOR scans give all 32 windows (nthash.hpp:100-119 restated).
__device__ __forceinline__ void compute_block(const WS& w, uint32_t Bp, uint64_t& fh, uint64_t& rh, uint32_t& pres, uint32_t& acc,
                              uint32_t& exist)
{
  const uint32_t lane = w.lane, k = w.k;
  const uint32_t a0 = Bp + lane, a1 = Bp + lane + 32;
  const uint32_t c0 = a0 < w.ve ? v_at(w, a0) : 0u;
  const uint32_t c1 = (a1 < w.ve && lane < 31) ? v_at(w, a1) : 0u;
  uint64_t u0 = srol(sF(w, c0), 62 - lane), u1 = lane < 31 ? srol(sF(w, c1), 30 - lane) : 0ull;
  uint64_t x0 = srol(sR(w, c0), lane), x1 = srol(sR(w, c1), lane + 32);
  u0 = xor_scan_incl(u0, lane); u1 = xor_scan_incl(u1, lane);
  x0 = xor_scan_incl(x0, lane); x1 = xor_scan_incl(x1, lane);
  u1 ^= __shfl_sync(kFull, u0, 31);
  x1 ^= __shfl_sync(kFull, x0, 31);
  // exclusive prefix at j (= inclusive at j-1) and inclusive prefix at j+k-1
  uint64_t pu = __shfl_up_sync(kFull, u0, 1), px = __shfl_up_sync(kFull, x0, 1);
  if (lane == 0) { pu = 0; px = 0; }
  const uint32_t e = lane + k - 1; // 0..62
  const uint64_t eu_lo = __shfl_sync(kFull, u0, e & 31u), eu_hi = __shfl_sync(kFull, u1, e & 31u);
  const uint64_t ex_lo = __shfl_sync(kFull, x0, e & 31u), ex_hi = __shfl_sync(kFull, x1, e & 31u);
  const uint64_t su = (e < 32 ? eu_lo : eu_hi) ^ pu;
  const uint64_t sx = (e < 32 ? ex_lo : ex_hi) ^ px;
  fh = sror(su, 63 - lane - k);
  rh = sror(sx, lane);
  const bool wexists = Bp + lane + k <= w.ve;
  const bool present = wexists && bf_contains(w, fh, rh);
  const uint32_t ca = Bp + k + lane;
  const bool cex = ca < w.ve;
  const bool cacc = cex && is_accepted(v_at(w, ca));
  pres = __ballot_sync(kFull, present);
  acc = __ballot_sync(kFull, cacc);
  exist = __ballot_sync(kFull, cex);
}

// ---- lane-0 rope surgery ---------------------------------------------------------------
struct Rope { // lane-0 view
  EdNode* nd;
  uint32_t nn, ncap;
  char* seq;
  uint32_t len;
  int err;
};
__device__ void rope_set(Rope& r, uint32_t i, const EdNode& v)
{ // "if (i < size) a[i] = v; else push_back(v)"
  if (i < r.nn) { st_node(r.nd + i, v); return; }
  if (i != r.nn || r.nn >= r.ncap) { r.err = 1; return; }
  st_node(r.nd + r.nn, v);
  r.nn++;
}
__device__ uint32_t rope_char(const Rope& r, uint32_t pos, uint32_t idx)
{
  if (idx >= r.nn) return 0;
  const EdNode n = ld_node(r.nd + idx);
  if (n.type == 0) return pos < r.len ? (unsigned char)r.seq[pos] : 0u;
  if (n.type == 1) return n.c;
  return 0;
}
__device__ void rope_increment(const Rope& r, uint32_t& pos, uint32_t& idx)
{
  if (idx >= r.nn) return;
  const EdNode n = ld_node(r.nd + idx);
  if (n.type == 0) {
    pos++;
    if (pos > n.e) {
      idx++;
      if (idx < r.nn) { const EdNode x = ld_node(r.nd + idx); if (x.type == 0) pos = x.s; }
    }
  } else if (n.type == 1) {
    idx++;
    if (idx < r.nn) { const EdNode x = ld_node(r.nd + idx); if (x.type == 0) pos = x.s; }
  }
}

// makeInsertion, :480-569
__device__ void rope_insert(Rope& r, uint32_t& t_idx, uint32_t insert_pos, const unsigned char* ins, uint32_t L)
{
  const EdNode orig = ld_node(r.nd + t_idx);
  if (orig.type == 0 && !(int(insert_pos) <= int(orig.s))) {
    EdNode head = orig;
    head.e = insert_pos - 1;
    st_node(r.nd + t_idx, head);
    for (uint32_t i = 0; i < L; i++) { EdNode c = { 1, 0, 0, ins[i] }; rope_set(r, t_idx + i + 1, c); }
    EdNode after = { 0, insert_pos, orig.e, 0 };
    rope_set(r, t_idx + L + 1, after);
    t_idx++;
    return;
  }
  if (orig.type == 0 || orig.type == 1) {
    // lift nodes [t_idx, t_idx+nre) up by L, then write the inserted characters
    uint32_t nre = 0;
    while (t_idx + nre < r.nn && ld_node(r.nd + t_idx + nre).type != -1) nre++;
    const uint32_t new_n = max(r.nn, t_idx + L + nre);
    if (new_n > r.ncap) { r.err = 1; return; }
    for (uint32_t q = nre; q > 0; q--) st_node(r.nd + t_idx + L + q - 1, ld_node(r.nd + t_idx + q - 1));
    r.nn = new_n;
    for (uint32_t q = 0; q < L; q++) { EdNode c = { 1, 0, 0, ins[q] }; st_node(r.nd + t_idx + q, c); }
  }
}

// makeDeletion, :574-664 (tail recursion unrolled)
__device__ void rope_delete(Rope& r, uint32_t& t_idx, uint32_t& pos, uint32_t num_del)
{
  for (;;) {
    if (t_idx >= r.nn) { r.err = 1; return; }
    const EdNode orig = ld_node(r.nd + t_idx);
    uint32_t leftover = 0;
    if (orig.type == 0) {
      if (pos <= orig.s) {
        if (pos + num_del <= orig.e) {
          EdNode n = orig; n.s = pos + num_del; st_node(r.nd + t_idx, n);
          pos = n.s;
          return;
        }
        leftover = pos + num_del - orig.e; // sic, :594
        pos = orig.e + 1;
        uint32_t i = t_idx + 1;
        while (i < r.nn) {
          EdNode x = ld_node(r.nd + i);
          if (x.type == -1) break;
          st_node(r.nd + i - 1, x);
          x.type = -1; st_node(r.nd + i, x);
          i++;
        }
      } else {
        if (pos + num_del <= orig.e) {
          EdNode split = { 0, pos + num_del, orig.e, 0 };
          EdNode n = orig; n.e = pos - 1; st_node(r.nd + t_idx, n);
          pos = split.s;
          t_idx++;
          rope_set(r, t_idx, split);
          return;
        }
        leftover = pos + num_del - orig.e; // sic, :622
        EdNode n = orig; n.e = pos - 1; st_node(r.nd + t_idx, n);
        pos = orig.e + 1;
        t_idx++;
      }
    } else if (orig.type == 1) {
      uint32_t i = t_idx;
      leftover = num_del;
      while (i < r.nn && leftover > 0) {
        EdNode x = ld_node(r.nd + i);
        if (x.type != 1) break;
        x.type = -1; st_node(r.nd + i, x);
        leftover--; i++;
      }
      uint32_t j = t_idx;
      while (i < r.nn) {
        EdNode x = ld_node(r.nd + i);
        if (x.type == -1) break;
        st_node(r.nd + j, x);
        x.type = -1; st_node(r.nd + i, x);
        i++; j++;
      }
    } else return;
    if (leftover == 0) return;
    if (!(t_idx < r.nn)) return;
    const EdNode nx = ld_node(r.nd + t_idx);
    if (nx.type == -1) return;
    if (nx.type == 0) pos = nx.s;
    num_del = leftover;
  }
}

// getPrevInsertion, :762-777
__device__ int rope_prev_insertion(const Rope& r, uint32_t t_seq, uint32_t t_idx, unsigned char* buf, int cap)
{
  int n = 0;
  uint32_t idx = t_idx;
  if (idx < r.nn) {
    const EdNode tn = ld_node(r.nd + idx);
    if ((tn.type == 0 && t_seq == tn.s) || tn.type == 1) idx--;
  }
  while (idx < r.nn) {
    const EdNode x = ld_node(r.nd + idx);
    if (x.type != 1) break;
    if (n < cap) buf[n] = rc_char(x.c);
    n++;
    idx--;
  }
  return n;
}

// isRepeatInsertion, :416-451
__device__ bool is_repeat(const unsigned char* s, int n)
{
  if (n <= 0 || n > 160) return false;
  int lps[160];
  lps[0] = 0;
  int len = 0, i = 1;
  while (i < n) {
    if (s[i] == s[len]) { len++; lps[i] = len; i++; }
    else if (len != 0) len = lps[len - 1];
    else { lps[i] = 0; i++; }
  }
  const int l = lps[n - 1];
  return l > 0 && n % (n - l) == 0;
}

// node shuffle of :1043-1056 / :1074-1088
__device__ void rope_remove_prev(Rope& r, uint32_t t_seq, uint32_t t_idx, uint32_t count)
{
  uint32_t j = 1;
  if (t_idx < r.nn) { const EdNode tn = ld_node(r.nd + t_idx); if (tn.type == 0 && t_seq == tn.s) j = 0; }
  for (uint32_t i = count; i > 0; i--) {
    if (i > t_idx) { r.err = 1; continue; }
    bool moved = false;
    if (t_idx + j < r.nn) {
      EdNode src = ld_node(r.nd + t_idx + j);
      if (src.type != -1) {
        st_node(r.nd + t_idx - i, src);
        src.type = -1; st_node(r.nd + t_idx + j, src);
        j++;
        moved = true;
      }
    }
    if (!moved) { EdNode x = ld_node(r.nd + t_idx - i); x.type = -1; st_node(r.nd + t_idx - i, x); }
  }
}

// findAcceptedKmer, :703-758.  kmer must hold 32 bytes.
__device__ bool rope_find_kmer(const Rope& r, uint32_t k, uint32_t& h_seq, uint32_t& t_seq, uint32_t& h_idx,
                               uint32_t& t_idx, unsigned char* kmer)
{
  uint32_t tt = t_idx, th = 0, i = t_seq, curr = t_idx;
  while (i < r.len && tt < r.nn && ld_node(r.nd + tt).type != -1) {
    uint32_t ch = rope_char(r, i, curr);
    if (is_accepted(ch)) {
      uint32_t kl = 0;
      kmer[kl++] = (unsigned char)ch;
      th = tt;
      uint32_t j = i;
      rope_increment(r, j, tt);
      while (j < r.len && tt < r.nn && ld_node(r.nd + tt).type != -1) {
        curr = tt;
        ch = rope_char(r, j, curr);
        if (!is_accepted(ch)) { i = j; break; }
        kmer[kl++] = (unsigned char)ch;
        if (kl == k) break;
        rope_increment(r, j, tt);
      }
      if (kl == k) { h_seq = i; t_seq = j; h_idx = th; t_idx = tt; return true; }
    }
    if (tt < r.nn) rope_increment(r, i, tt); else break;
  }
  h_seq = r.len; t_seq = r.len;
  return false;
}

// i-th string of multi_possible_bases[first] (:198-343): length-major, A<C<G<T
__device__ __forceinline__ uint32_t insertion_string(uint32_t first, uint32_t i, unsigned char* out)
{
  const uint32_t L = i < 1 ? 1 : i < 5 ? 2 : i < 21 ? 3 : i < 85 ? 4 : 5;
  const uint32_t start = L == 1 ? 0 : L == 2 ? 1 : L == 3 ? 5 : L == 4 ? 21 : 85;
  uint32_t r = i - start;
  out[0] = (unsigned char)first;
  for (uint32_t p = L - 1; p >= 1; p--) {
    const uint32_t d = r & 3u;
    out[p] = d == 0 ? 'A' : d == 1 ? 'C' : d == 2 ? 'G' : 'T';
    r >>= 2;
  }
  return L;
}
__device__ __forceinline__ uint32_t num_tries(uint32_t max_ins)
{ // :150
  return max_ins == 0 ? 0 : max_ins == 1 ? 1 : max_ins == 2 ? 5 : max_ins == 3 ? 21 : max_ins == 4 ? 85 : 341;
}
// polish_bases_array, :158-174, packed little-endian into one word; returns the count
__device__ __forceinline__ uint32_t polish_bases(uint32_t draft, uint32_t& packed)
{
#define GP_P3(a, b, c) (uint32_t(a) | (uint32_t(b) << 8) | (uint32_t(c) << 16))
  switch (draft) {
  case 'A': packed = GP_P3('T', 'C', 'G'); return 3;
  case 'T': packed = GP_P3('A', 'C', 'G'); return 3;
  case 'C': packed = GP_P3('A', 'T', 'G'); return 3;
  case 'G': packed = GP_P3('A', 'T', 'C'); return 3;
  case 'R': packed = GP_P3('T', 'C', 0); return 2;
  case 'Y': packed = GP_P3('A', 'G', 0); return 2;
  case 'S': packed = GP_P3('A', 'T', 0); return 2;
  case 'W': packed = GP_P3('C', 'G', 0); return 2;
  case 'K': packed = GP_P3('A', 'C', 0); return 2;
  case 'M': packed = GP_P3('T', 'G', 0); return 2;
  case 'B': packed = 'A'; return 1;
  case 'D': packed = 'C'; return 1;
  case 'H': packed = 'G'; return 1;
  case 'V': packed = 'T'; return 1;
  case 'N': packed = GP_P3('A', 'T', 'C') | (uint32_t('G') << 24); return 4;
  default: packed = 0; return 0;
  }
#undef GP_P3
}

struct Best {
  uint32_t type;    // 0 none, 1 substitution, 2 insertion, 3 deletion
  uint32_t support;
  uint32_t sub_base;
  uint32_t ins_first, ins_index; // insertion string = insertion_string(ins_first, ins_index)
  uint32_t del_len;
};

constexpr uint32_t kInsZeroRow = 4u * 3u * 32u; // w.insF / w.insR: twelve rows of terms, then a row of zeros

// tryIndels + tryDeletion, :1157-1411.  Lanes share the candidates; the reference's visiting
// order (ins_0, del_0, ins_1, del_1, ..., ins_340) breaks support ties, later wins (:1347,:1384).
__device__ __forceinline__ bool try_indels(WS& w, uint32_t draft_char, uint32_t index_char, uint32_t& num_deletions, Best& best)
{
  const uint32_t ntry = num_tries(w.max_ins);
  const uint32_t k = w.k;
  const uint32_t an = ahead_count(w);
  uint32_t best_key = 0; // (support << 12) | order+1 for modes 1/2; mode 0 keeps the smallest order
  uint32_t first_key = 0xffffffffu;
  uint32_t ndel = 0;     // deletions num_deletions .. max_del, one per visited insertion index (:1359-1396)
  // Stage what every candidate shares: the outgoing bases E[h..t-1] (their k-rotated forward
  // seed and plain reverse seed) and the incoming bases ahead of t (plain forward, k-rotated
  // reverse), so that one roll is four shared-memory loads and a handful of logic ops.
  {
    uint64_t* outF = w.stage, *outR = w.stage + 32, *inF = w.stage + 64, *inRk = w.stage + 128;
    __syncwarp();
    if (w.lane + 1 < k) {
      const uint32_t c = ring_at(w, w.lane);
      outF[w.lane] = w.seedt[8 + w.code[c]];
      outR[w.lane] = w.seedt[16 + (c & 7u)];
    }
    for (uint32_t q = w.lane; q < 64; q += 32) {
      const uint32_t c = q < an ? ahead_at(w, q) : 0u;
      inF[q] = w.seedt[w.code[c]];
      inRk[q] = w.seedt[24 + (c & 7u)];
    }
    __syncwarp();
    HashState base = w.hs;
    ws_changelast(w, base, draft_char, index_char); // :1290
    const uint64_t dF = w.seedt[w.code[draft_char]], dRk = w.seedt[24 + (draft_char & 7u)];
    // a candidate can no longer qualify once it has missed more samples than the threshold allows
    const uint32_t nsamp = (k - 2) / w.jump + 1;
    const uint32_t need = w.thrE > 0.0f ? (uint32_t)ceilf(w.thrE) : 0u;
    const uint32_t allowed = nsamp >= need ? nsamp - need : 0u;
    // No candidate is rolled.  ntHash is XOR-linear in the characters of the window, so the hashes of a candidate's
    // windows are those of the "all-A" candidate of the same length (the COMMON chain: one lane per length rolls it
    // once, k-1 steps) XOR one precomputed term per inserted base that is not an A (w.insF / w.insR: the seed
    // difference rotated by the distance between the base's entry and the sampled roll).  A lane takes a GROUP of four
    // candidates that differ in their last inserted base only: the common hash and the terms of the bases they share
    // are fetched once per sample, and only sampled rolls are ever looked at.  The 16 filter words of a sample are in
    // flight together and are consumed one sample later.
    //
    // The deletion candidates (:1359-1396, tryDeletion :1157-1234) ARE rolled -- there are at most ten of them -- in the
    // same loop as the common chains, on lanes of their own (8 + i), their filter words pending across the rolls.
    uint64_t* comF = w.com, *comR = w.com + 5 * 32;
    if (num_deletions <= w.max_del) ndel = min(ntry, w.max_del - num_deletions + 1);
    {
      const bool role_c = w.lane < w.max_ins;
      const bool role_d = w.lane >= 8u && w.lane < 8u + ndel;
      const uint32_t L = w.lane + 1;                       // role C
      const uint32_t nd = num_deletions + (w.lane - 8u);   // role D: bases deleted
      HashState t = role_d ? w.hs : base;
      bool d_act = false, d_pend = false;
      uint32_t d_present = 0, d_pb = 0, d_pw[4] = { 0, 0, 0, 0 };
      auto d_issue = [&]() {
        const uint64_t bb = t.fh + t.rh;
        uint64_t h1 = bb * w.mul1, h2 = bb * w.mul2, h3 = bb * w.mul3;
        h1 ^= h1 >> kMultiShift; h2 ^= h2 >> kMultiShift; h3 ^= h3 >> kMultiShift;
        const uint32_t n0 = bf_index(bb), n1 = bf_index(h1), n2 = bf_index(h2), n3 = bf_index(h3);
        d_pw[0] = ld_filter(w.bf + (n0 >> 5)); d_pw[1] = ld_filter(w.bf + (n1 >> 5));
        d_pw[2] = ld_filter(w.bf + (n2 >> 5)); d_pw[3] = ld_filter(w.bf + (n3 >> 5));
        d_pb = (n0 & 31u) | ((n1 & 31u) << 8) | ((n2 & 31u) << 16) | ((n3 & 31u) << 24);
        d_pend = true;
      };
      auto d_consume = [&]() {
        if (d_pend && ((d_pw[0] >> (d_pb & 31u)) & (d_pw[1] >> ((d_pb >> 8) & 31u)) & (d_pw[2] >> ((d_pb >> 16) & 31u)) &
                       (d_pw[3] >> (d_pb >> 24)) & 1u) != 0u) d_present++;
        d_pend = false;
      };
      if (role_d && nd - 1 < an) { // the character that follows the deleted run must exist
        ws_changelast(w, t, draft_char, ahead_at(w, nd - 1)); // :1190-1197
        d_act = true;
        d_issue();                                             // the first k-mer always counts (:1201-1203)
      }
      for (uint32_t kk = 0; kk + 1 < k; kk++) {
        if (role_c) { // :1294-1326 with A for every inserted base after the first
          uint64_t inf, inr;
          if (kk + 1 < L) { inf = w.seedt[1]; inr = w.seedt[24 + 1]; }
          else if (kk + 1 == L) { inf = dF; inr = dRk; }   // then the draft base (:1279)
          else { inf = inF[kk - L]; inr = inRk[kk - L]; }
          t.fh = srol1(t.fh) ^ inf ^ outF[kk];
          t.rh = sror1(t.rh ^ inr ^ outR[kk]);
          comF[w.lane * 32 + kk] = t.fh;
          comR[w.lane * 32 + kk] = t.rh;
        } else if (d_act && kk + 2 < k) { // roll kk + 1 of :1204-1220
          const uint32_t ai = nd + kk;
          if (ai >= an) d_act = false; // roll() fails: end of contig
          else {
            t.fh = srol1(t.fh) ^ inF[ai] ^ outF[kk];
            t.rh = sror1(t.rh ^ inRk[ai] ^ outR[kk]);
            if ((w.samp >> (kk + 1)) & 1ull) { d_consume(); d_issue(); }
          }
        }
      }
      d_consume();
      if (role_d && float(d_present) >= w.thrD && d_present > 0) { // :1226-1233 (returns 0 when rejected)
        const uint32_t order = 2 * (w.lane - 8u) + 1;
        const uint32_t key = (d_present << 12) | (order + 1);
        best_key = max(best_key, key);
        first_key = min(first_key, order);
      }
    }
    __syncwarp();
    // groups, longest strings first: 64 of length 5 (three shared bases), 16 of length 4, 4 of length 3, one of
    // length 2 (its four candidates share nothing but the first base) and the single string of length 1
    const uint32_t n5 = w.max_ins >= 5 ? 64u : 0u, n4 = w.max_ins >= 4 ? 16u : 0u, n3 = w.max_ins >= 3 ? 4u : 0u,
                   n2 = w.max_ins >= 2 ? 1u : 0u, n1 = w.max_ins >= 1 ? 1u : 0u;
    const uint32_t n_groups = n5 + n4 + n3 + n2 + n1;
    constexpr int G = 4;
    for (uint32_t g0 = 0; g0 < n_groups; g0 += 32) {
      const uint32_t g = g0 + w.lane;
      uint32_t L = 0, pre = 0;
      if (g < n5) { L = 5; pre = g; }
      else if (g < n5 + n4) { L = 4; pre = g - n5; }
      else if (g < n5 + n4 + n3) { L = 3; pre = g - n5 - n4; }
      else if (g < n5 + n4 + n3 + n2) { L = 2; }
      else if (g < n_groups) { L = 1; }
      const uint32_t start = L == 1 ? 0u : L == 2 ? 1u : L == 3 ? 5u : L == 4 ? 21u : 85u; // index of the class's first string
      // table rows of the shared bases (string positions 1 .. L-2 enter at rolls 0 .. L-3); an A has no term: row of zeros
      uint32_t row[3];
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const uint32_t d = (L >= 3u + j) ? (pre >> (2u * (L - 3u - j))) & 3u : 0u;
        row[j] = d ? (uint32_t(j) * 3u + d - 1u) * 32u : kInsZeroRow;
      }
      const uint32_t last_row = L >= 2 ? (L - 2u) * 3u * 32u : 0u; // rows of the last inserted base (enters at roll L-2)
      const uint32_t com_row = L ? (L - 1u) * 32u : 0u;
      // Two samples are in flight (buffers A and B): the words of sample s+1 are requested before those of sample s are
      // looked at, so that the L2 latency hides behind the hashing of the next sample.  Nothing below branches on a
      // candidate -- a candidate that can no longer qualify keeps being hashed (its words are valid addresses) and
      // only the warp-wide vote ends the loop -- so that the four candidates' chains interleave.
      uint32_t presq[G], missq[G], pbA[G], pwA[G][4], pbB[G], pwB[G][4];
#pragma unroll
      for (int q = 0; q < G; q++) { presq[q] = 0; missq[q] = 0; }
      auto issue = [&](uint32_t kk, uint32_t (&pw)[G][4], uint32_t (&pb)[G]) {
        uint64_t pf = comF[com_row + kk], pr = comR[com_row + kk];
#pragma unroll
        for (int j = 0; j < 3; j++) { pf ^= w.insF[row[j] + kk]; pr ^= w.insR[row[j] + kk]; }
#pragma unroll
        for (int q = 0; q < G; q++) {
          uint64_t f = pf, r = pr;
          if (q) { f ^= w.insF[last_row + uint32_t(q - 1) * 32u + kk]; r ^= w.insR[last_row + uint32_t(q - 1) * 32u + kk]; }
          const uint64_t b = f + r;
          uint64_t h1 = b * w.mul1, h2 = b * w.mul2, h3 = b * w.mul3;
          h1 ^= h1 >> kMultiShift; h2 ^= h2 >> kMultiShift; h3 ^= h3 >> kMultiShift;
          const uint32_t n0 = bf_index(b), n1 = bf_index(h1), n2 = bf_index(h2), n3 = bf_index(h3);
          pw[q][0] = ld_filter(w.bf + (n0 >> 5)); pw[q][1] = ld_filter(w.bf + (n1 >> 5));
          pw[q][2] = ld_filter(w.bf + (n2 >> 5)); pw[q][3] = ld_filter(w.bf + (n3 >> 5));
          pb[q] = (n0 & 31u) | ((n1 & 31u) << 8) | ((n2 & 31u) << 16) | ((n3 & 31u) << 24);
        }
      };
      auto consume = [&](const uint32_t (&pw)[G][4], const uint32_t (&pb)[G]) {
#pragma unroll
        for (int q = 0; q < G; q++) {
          const uint32_t hit = (pw[q][0] >> (pb[q] & 31u)) & (pw[q][1] >> ((pb[q] >> 8) & 31u)) &
                               (pw[q][2] >> ((pb[q] >> 16) & 31u)) & (pw[q][3] >> (pb[q] >> 24)) & 1u;
          presq[q] += hit;
          missq[q] += hit ^ 1u;
        }
      };
      // a candidate that has missed more samples than the threshold allows cannot qualify (its support stays below
      // ceil(thrE) whatever the remaining samples say): once no lane holds a live one the group is settled
      auto live = [&]() {
        bool a = false;
#pragma unroll
        for (int q = 0; q < G; q++) a |= (L >= 2 || (L == 1 && q == 0)) && missq[q] <= allowed;
        return __any_sync(kFull, a);
      };
      // the sampled rolls only (kk % jump == 0, :1294-1310): kk = 0, jump, 2 jump .. < k - 1
      uint32_t kk = 0;
      issue(kk, pwA, pbA);
      kk += w.jump;
      for (;;) {
        const bool moreB = kk + 1 < k;
        if (moreB) issue(kk, pwB, pbB);
        kk += w.jump;
        consume(pwA, pbA);
        if (!moreB || !live()) break;
        const bool moreA = kk + 1 < k;
        if (moreA) issue(kk, pwA, pbA);
        kk += w.jump;
        consume(pwB, pbB);
        if (!moreA || !live()) break;
      }
#pragma unroll
      for (int q = 0; q < G; q++) {
        const bool exists = L >= 2 || (L == 1 && q == 0);
        const uint32_t i = start + pre * 4u + uint32_t(q); // position in multi_possible_bases[first] (:198-343)
        if (exists && missq[q] <= allowed && i < ntry && float(presq[q]) >= w.thrE && (w.mode == 0 || presq[q] > 0)) { // :1333-1337, :1400
          const uint32_t order = 2 * i;
          const uint32_t key = (presq[q] << 12) | (order + 1);
          best_key = max(best_key, key);
          first_key = min(first_key, order);
        }
      }
    }
  }
  num_deletions += ndel;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    best_key = max(best_key, __shfl_xor_sync(kFull, best_key, o));
    first_key = min(first_key, __shfl_xor_sync(kFull, first_key, o));
  }
  if (best_key == 0 && first_key == 0xffffffffu) return false;
  uint32_t order, support;
  if (w.mode == 0) { // first good indel wins (:1338-1344, :1377-1382); its support is only recorded
    order = first_key;
    support = 1;
  } else {
    order = (best_key & 0xfffu) - 1;
    support = best_key >> 12;
  }
  if (w.mode == 2 && !(support > best.support)) return true; // :1401
  if (order & 1u) { best.type = 3; best.del_len = (num_deletions - ndel) + (order >> 1); }
  else { best.type = 2; best.ins_first = index_char; best.ins_index = order >> 1; }
  best.support = support;
  return true;
}

// makeEdit, :972-1154
__device__ __forceinline__ void make_edit(WS& w, uint32_t draft_char, const Best& best)
{
  const uint32_t k = w.k;
  if (best.type == 0) {
    // no fix found (:1131-1146): soft-mask the base when -a1.  The rope shape, both cursors and
    // every window hash are unchanged, so this touches nothing but the character itself.
    if (w.mask) {
      const uint32_t lc = to_lower(draft_char);
      if (w.t.n.type == 0) { if (w.lane == 0) w.seq[w.t.pos] = (char)lc; }
      else if (w.t.n.type == 1) { w.t.n.c = lc; if (w.lane == 0) st_node(w.nd + w.t.idx, w.t.n); }
      w.n_mask++;
    }
    return;
  }
  uint32_t new_last = 0;   // character now sitting at the tail of the window
  bool stream_changed = false, reseeded = false, found = false;
  unsigned char* kmer = w.kmer;
  if (w.lane == 0) {
    Rope r = { w.nd, w.nn, w.ncap, w.seq, w.len, 0 };
    uint32_t t_idx = w.t.idx, t_seq = w.t.pos, h_idx = w.h.idx, h_seq = w.h.pos;
    const EdNode tn = ld_node(r.nd + t_idx);
    switch (best.type) {
    case 1: // :1002-1033
      if (tn.type == 0) r.seq[t_seq] = (char)best.sub_base;
      else if (tn.type == 1) { EdNode x = tn; x.c = best.sub_base; st_node(r.nd + t_idx, x); }
      new_last = best.sub_base;
      break;
    case 2: { // :1034-1115
      unsigned char ins[8];
      const uint32_t L = insertion_string(best.ins_first, best.ins_index, ins);
      unsigned char prev[176];
      int np = rope_prev_insertion(r, t_seq, t_idx, prev, 160);
      if (np > 160) { r.err = 1; np = 160; }
      bool skipped = false;
      if (uint32_t(np) + L >= k) {
        if (is_repeat(prev, np) || uint32_t(np) + L >= w.icap) {
          rope_remove_prev(r, t_seq, t_idx, uint32_t(np));
          found = rope_find_kmer(r, k, h_seq, t_seq, h_idx, t_idx, kmer);
          skipped = true;
        } else {
          for (uint32_t x = 0; x < L; x++) { // :1070-1100
            for (int q = np; q > 0; q--) prev[q] = prev[q - 1];
            prev[0] = rc_char(ins[x]);
            np++;
            if (is_repeat(prev, np)) {
              rope_remove_prev(r, t_seq, t_idx, uint32_t(np) - x);
              found = rope_find_kmer(r, k, h_seq, t_seq, h_idx, t_idx, kmer);
              skipped = true;
            }
          }
        }
      }
      if (skipped) { reseeded = true; break; }
      rope_insert(r, t_idx, t_seq, ins, L);
      new_last = ins[0];
      stream_changed = true;
      break;
    }
    case 3: // :1116-1130
      rope_delete(r, t_idx, t_seq, best.del_len);
      new_last = rope_char(r, t_seq, t_idx);
      stream_changed = true;
      break;
    default: // :1131-1146
      if (w.mask) {
        const uint32_t lc = to_lower(draft_char);
        if (tn.type == 0) r.seq[t_seq] = (char)lc;
        else if (tn.type == 1) { EdNode x = tn; x.c = lc; st_node(r.nd + t_idx, x); }
        new_last = lc;
      } else new_last = draft_char;
      break;
    }
    w.nn = r.nn;
    w.err |= r.err;
    w.t.idx = t_idx; w.t.pos = t_seq; w.h.idx = h_idx; w.h.pos = h_seq;
  }
  __syncwarp();
  w.nn = __shfl_sync(kFull, w.nn, 0);
  w.err = __shfl_sync(kFull, w.err, 0);
  w.t.idx = __shfl_sync(kFull, w.t.idx, 0);
  w.t.pos = __shfl_sync(kFull, w.t.pos, 0);
  w.h.idx = __shfl_sync(kFull, w.h.idx, 0);
  w.h.pos = __shfl_sync(kFull, w.h.pos, 0);
  new_last = __shfl_sync(kFull, new_last, 0);
  stream_changed = __shfl_sync(kFull, int(stream_changed), 0) != 0;
  reseeded = __shfl_sync(kFull, int(reseeded), 0) != 0;
  found = __shfl_sync(kFull, int(found), 0) != 0;
  cur_load(w, w.t);
  cur_load(w, w.h);
  w.blk_valid = false; // the window's last character changed: every cached hash is stale
  if (reseeded) {
    w.n_roll++;
    if (found && w.lane < k) w.vb[(w.hp + w.lane) & (kVBuf - 1)] = kmer[w.lane]; // window the reference re-seeded from
    w.ve = w.hp + k; w.exhausted = false; w.m = w.t;
    __syncwarp();
    return;
  }
  if (w.lane == 0) w.vb[(w.hp + k - 1) & (kVBuf - 1)] = (unsigned char)new_last;
  w.n_edit++;
  if (stream_changed) { w.ve = w.hp + k; w.exhausted = false; w.m = w.t; }
  __syncwarp();
}

// One contig through one k: kmerizeAndCorrect, :1414-1771.  Result is left in the rope.
__device__ __forceinline__ void edit_round(WS& w)
{
  const uint32_t k = w.k, lane = w.lane, len = w.len;
  if (len == 0) { w.nn = 0; return; }
  // findFirstAcceptedKmer(0), :392-413: smallest i with [i, i+k) accepted and i + k < len
  uint32_t h0 = len - 1;
  {
    uint32_t run = 0;
    bool found = false;
    for (uint32_t base = 0; base + 1 < len && !found; base += 32) {
      const uint32_t e = base + lane;
      const bool a = (e + 1 < len) && is_accepted((unsigned char)w.seq[e]);
      const uint32_t bits = __ballot_sync(kFull, a);
      if (bits == 0xffffffffu && run + 32 < k) { run += 32; continue; }
      for (uint32_t i = 0; i < 32; i++) {
        if ((bits >> i) & 1u) { run++; if (run >= k) { h0 = base + i + 1 - k; found = true; break; } }
        else run = 0;
      }
    }
  }
  // root node (:1451-1456)
  if (lane == 0) { EdNode root = { 0, 0, len - 1, 0 }; st_node(w.nd, root); }
  w.nn = 1;
  __syncwarp();
  if (uint64_t(h0) + k - 1 >= len) return; // no seed: the do-loop breaks at once (:1463)
  // seed window (:1441-1444); absolute stream indices start at the draft position
  w.hp = h0;
  if (lane < k) w.vb[(h0 + lane) & (kVBuf - 1)] = (unsigned char)w.seq[h0 + lane];
  w.ve = h0 + k;
  w.exhausted = false;
  w.h.pos = h0; w.h.idx = 0; cur_load(w, w.h);
  w.t.pos = h0 + k - 1; w.t.idx = 0; cur_load(w, w.t);
  w.m = w.t;
  w.blk_valid = false;
  // seed tables for this k (nthash.hpp:21-63): plain and rotated by k, both strands
  if (lane < 5) {
    const uint64_t f = lane == 0 ? 0ull : seed_of_code(lane - 1);
    w.seedt[lane] = f;
    w.seedt[8 + lane] = srol(f, k);
  }
  if (lane >= 8 && lane < 16) {
    const uint64_t r = cseed_of_char(lane - 8);
    w.seedt[16 + lane - 8] = r;
    w.seedt[24 + lane - 8] = srol(r, k);
  }
  __syncwarp();
  // insertion-search terms: an inserted base d (instead of A) that enters at roll j shows up in the hash after roll kk
  // as its seed difference rotated by the rolls in between (forward: kk - j; reverse, on the k-rotated seed: kk - j + 1)
  {
    uint64_t* tF = const_cast<uint64_t*>(w.insF);
    uint64_t* tR = const_cast<uint64_t*>(w.insR);
    for (uint32_t e = lane; e < 4u * 3u * 32u; e += 32) {
      const uint32_t kk = e & 31u, jd = e >> 5, j = jd / 3u, d = jd - 3u * j + 1u;
      const uint64_t df = w.seedt[1 + d] ^ w.seedt[1];
      const uint64_t dr = w.seedt[24 + ((0x4731u >> (4 * d)) & 7u)] ^ w.seedt[24 + 1];
      tF[e] = kk >= j ? srol(df, kk - j) : 0ull;
      tR[e] = kk >= j ? sror(dr, kk - j + 1u) : 0ull;
    }
    tF[kInsZeroRow + lane] = 0ull; // the row an inserted A points at
    tR[kInsZeroRow + lane] = 0ull;
  }
  w.samp = 0;
  for (uint32_t kk = 0; kk < k; kk += w.jump) w.samp |= 1ull << kk;
  const uint64_t kbits = k >= 64 ? ~0ull : ((1ull << k) - 1ull);
  __syncwarp();

  for (;;) {
    if (w.err) return;
    if (uint64_t(w.h.pos) + k - 1 >= len) break; // :1463
    if (!w.blk_valid) {
      w.B = w.hp;
      stream_fill(w, w.B + 106);
      uint32_t p0, a0, e0, p1, a1, e1;
      compute_block(w, w.B, w.f0, w.r0, p0, a0, e0);
      compute_block(w, w.B + 32, w.f1, w.r1, p1, a1, e1);
      w.pres = uint64_t(p0) | (uint64_t(p1) << 32);
      w.acc = uint64_t(a0) | (uint64_t(a1) << 32);
      w.exist = uint64_t(e0) | (uint64_t(e1) << 32);
      w.blk_valid = true;
    }
    uint32_t j = w.hp - w.B;
    if (j >= 32) {
      if (j >= 64) { w.blk_valid = false; continue; }
      w.f0 = w.f1; w.r0 = w.r1;
      w.pres >>= 32; w.acc >>= 32; w.exist >>= 32;
      w.B += 32; j -= 32;
      stream_fill(w, w.B + 106);
      uint32_t p1, a1, e1;
      compute_block(w, w.B + 32, w.f1, w.r1, p1, a1, e1);
      w.pres |= uint64_t(p1) << 32; w.acc |= uint64_t(a1) << 32; w.exist |= uint64_t(e1) << 32;
    }
    // ---- scan the rest of block 0: first absent window, non-accepted incoming base or end ----
    const uint32_t span = 32 - j;
    const uint64_t evbits = ((~w.pres | ~w.acc) >> j) & (span >= 64 ? ~0ull : ((1ull << span) - 1ull));
    const uint32_t adv = evbits ? uint32_t(__ffsll((long long)evbits) - 1) : span;
    if (adv) {
      cur_advance(w, w.h, adv);
      cur_advance(w, w.t, adv);
      w.hp += adv;
      j += adv;
    }
    if (!evbits) continue;
    if (uint64_t(w.h.pos) + k - 1 >= len) break; // loop-top check of the iteration we landed on

    if (!((w.pres >> j) & 1ull)) {
      // ---- run of absent windows: speculate that the next positions end in "no fix" ----
      // A soft-mask changes no hash, so for up to 10 consecutive positions the look-ahead
      // counts come from the cached bits and all their candidate gates (:1565-1570) are
      // looked up in ONE phase (lane = 3 * position + candidate).  Positions are then
      // committed in order until one needs the full search, a skip, or the end of the block.
      {
        const uint32_t g = lane / 3u, bsel = lane - 3u * g, wj = j + g;
        const bool in_range = lane < 30u && wj < 32u;
        const uint32_t wjc = wj & 31u;
        bool attempt_l = false;
        if (in_range && !((w.pres >> wjc) & 1ull) && (((w.acc >> wjc) & kbits) == kbits))
          attempt_l = float((uint32_t)__popcll((~w.pres >> (wjc + 1)) & w.samp)) >= w.thrM;
        const uint32_t dch = to_upper(v_at(w, w.hp + g + k - 1));
        uint32_t pk;
        const uint32_t nbl = polish_bases(dch, pk);
        HashState gh;
        gh.fh = __shfl_sync(kFull, w.f0, wjc);
        gh.rh = __shfl_sync(kFull, w.r0, wjc);
        bool gate_l = false;
        if (attempt_l && bsel < nbl) {
          if (w.mode == 2) gate_l = true;
          else { ws_changelast(w, gh, dch, (pk >> (8 * bsel)) & 255u); gate_l = bf_contains(w, gh); }
        }
        const uint32_t gate_bits = __ballot_sync(kFull, gate_l);
        uint32_t done = 0;
        // commit: lane s decides position j+s; the run ends at the first position that needs
        // the full search, a skip, the end of the block or the end of the contig
        bool absent_s = false, att_s = false, stop_s = lane >= 10u;
        if (lane < 10u) {
          const uint32_t wq = j + lane;
          stop_s = wq >= 32u || !((w.acc >> (wq & 63u)) & 1ull) || uint64_t(w.h.pos) + lane + k - 1 >= len;
          if (!stop_s) {
            absent_s = !((w.pres >> wq) & 1ull);
            att_s = absent_s && (((w.acc >> wq) & kbits) == kbits) &&
                    float((uint32_t)__popcll((~w.pres >> (wq + 1)) & w.samp)) >= w.thrM;
            stop_s = att_s && ((gate_bits >> (3 * lane)) & 7u) != 0u; // a candidate is present: full search
          }
        }
        const uint32_t n_run = uint32_t(__ffs(__ballot_sync(kFull, stop_s))) - 1u; // <= 10
        const bool in_nodes = w.h.n.type == 0 && w.t.n.type == 0 && w.h.pos + n_run <= w.h.n.e &&
                              w.t.pos + n_run <= w.t.n.e;
        if (in_nodes) {
          // both cursors stay inside their draft ranges: all positions of the run at once
          const bool mine = lane < n_run;
          if (mine && att_s && w.mask)
            w.seq[w.t.pos + lane] = (char)to_lower(to_upper(v_at(w, w.hp + lane + k - 1))); // :1131-1146
          w.n_trig += __popc(__ballot_sync(kFull, mine && absent_s));
          if (w.mask) w.n_mask += __popc(__ballot_sync(kFull, mine && att_s));
          w.h.pos += n_run; w.t.pos += n_run; w.hp += n_run;
          done = n_run;
        } else {
          for (uint32_t s2 = 0; s2 < n_run; s2++) {
            const uint32_t wq = j + s2;
            if (uint64_t(w.h.pos) + k - 1 >= len) break; // :1463 with the real head cursor
            if (!((w.pres >> wq) & 1ull)) {
              const bool att = (((w.acc >> wq) & kbits) == kbits) &&
                               float((uint32_t)__popcll((~w.pres >> (wq + 1)) & w.samp)) >= w.thrM;
              if (att) {
                Best none = { 0, 0, 0, 0, 0, 0 };
                make_edit(w, to_upper(v_at(w, w.hp + k - 1)), none);
              }
              w.n_trig++;
            }
            cur_increment(w, w.h);
            cur_increment(w, w.t);
            w.hp++;
            done++;
          }
        }
        if (done) continue;
      }
      // ---- the window is absent: look-ahead confirmation (:1470-1523) ----
      w.n_trig++;
      const uint32_t draft_char = to_upper(ring_at(w, k - 1)); // :1480
      const bool all_ok = ((w.acc >> j) & kbits) == kbits;      // k more accepted bases exist
      if (all_ok) {
        const uint32_t check_missing = (uint32_t)__popcll((~w.pres >> (j + 1)) & w.samp);
        if (float(check_missing) >= w.thrM) { // :1517-1523
          w.hs.fh = __shfl_sync(kFull, w.f0, j);
          w.hs.rh = __shfl_sync(kFull, w.r0, j);
          uint32_t num_deletions = 1;       // :1526
          Best best = { 0, 0, 0, 0, 0, 0 };
          uint32_t packed;
          const uint32_t nb = polish_bases(draft_char, packed);
          // gate: is the k-mer ending in the candidate base present? (:1565-1570)
          HashState g = w.hs;
          const uint32_t my_base = (packed >> (8 * (lane & 3u))) & 255u;
          ws_changelast(w, g, draft_char, my_base);
          const bool gate = lane < nb && (w.mode == 2 || bf_contains(w, g));
          const uint32_t gates = __ballot_sync(kFull, gate);
          if (gates) {
            // windows j+1 .. j+k of the unedited stream, lane i <- window j+1+i
            const uint32_t wi = j + 1 + lane; // <= 63 for lane < k
            const uint64_t bf_lo = __shfl_sync(kFull, w.f0, wi & 31u), bf_hi = __shfl_sync(kFull, w.f1, wi & 31u);
            const uint64_t br_lo = __shfl_sync(kFull, w.r0, wi & 31u), br_hi = __shfl_sync(kFull, w.r1, wi & 31u);
            const uint64_t base_f = wi < 32 ? bf_lo : bf_hi, base_r = wi < 32 ? br_lo : br_hi;
            for (uint32_t b = 0; b < nb; b++) {
              if (!((gates >> b) & 1u)) continue;
              const uint32_t sub_base = (packed >> (8 * b)) & 255u;
              // replacing the tail base changes window j+1+i by one rotated seed difference per
              // strand (:1585-1606); window j+k no longer contains the base
              uint64_t cf = base_f, cr = base_r;
              if (lane + 1 < k) {
                cf ^= srol(sF(w, draft_char) ^ sF(w, sub_base), 1 + lane);
                cr ^= srol(sR(w, draft_char) ^ sR(w, sub_base), k - 2 - lane);
              }
              const bool hit = ((w.samp >> lane) & 1ull) && bf_contains(w, cf, cr); // lane < k && lane % jump == 0
              const uint32_t present = __popc(__ballot_sync(kFull, hit));
              if (float(present) >= w.thrE) { // :1621-1626
                if (present >= best.support) { best.type = 1; best.sub_base = sub_base; best.support = present; }
                if (w.mode == 0 || w.mode == 1) continue; // :1680-1682
              }
              if (w.mode == 2 || best.type != 1) { // :1686
                if (try_indels(w, draft_char, sub_base, num_deletions, best)) {
                  if (w.mode == 0 || w.mode == 1) break; // :1707-1709
                }
              }
            }
            // a substitution trial was made and reverted with the UPPER-cased base (:1609-1615)
            if (w.t.n.type == 0) { if (lane == 0) w.seq[w.t.pos] = (char)draft_char; }
            else if (w.t.n.type == 1) { w.t.n.c = draft_char; if (lane == 0) st_node(w.nd + w.t.idx, w.t.n); }
            __syncwarp();
          }
          make_edit(w, draft_char, best); // :1715-1736
          if (w.err) return;
        }
      }
    }
    // ---- roll forward, skipping k past any non-accepted incoming character (:1740-1759) ----
    long long target = -1;
    bool alive = true;
    do {
      if (cur_dead(w, w.h)) { alive = false; break; }      // roll(), :952
      stream_fill(w, w.hp + k + 1);
      cur_increment(w, w.h);
      if (cur_dead(w, w.t) || w.ve <= w.hp + k) { alive = false; break; } // :958-965
      const uint32_t in = v_at(w, w.hp + k);
      cur_increment(w, w.t);
      w.hp++;
      if (!is_accepted(in)) target = (long long)w.t.pos + (long long)k;
    } while (target >= 0 && (long long)w.t.pos != target);
    if (!alive) break;
  }
}

// writeEditsToFile body (:797-935): walk the rope until the first unset node.  kTrack: every emitted byte also gets its
// origin -- a draft range's bytes take the origins of the input bytes they copy, an inserted byte GP_EDIT_INSERTED -- so
// that the map to the original draft is composed over the k chain as the bytes are copied.  A template parameter, not
// a pointer test: the default instantiation is the kernel without tracking, instruction for instruction.
template<bool kTrack>
__device__ __forceinline__ uint32_t emit_rope(const WS& w, char* dst, uint32_t cap, int& err, const uint32_t* oin, uint32_t* oout)
{
  uint32_t o = 0;
  for (uint32_t i = 0; i < w.nn; i++) {
    const EdNode n = ld_node(w.nd + i);
    if (n.type == -1) break;
    if (n.type == 0) {
      if (n.s > w.len) continue; // substr would throw; never reached in valid runs
      uint32_t cnt = (n.e + 1u >= n.s) ? (n.e + 1u - n.s) : (w.len - n.s);
      if (n.s + cnt > w.len) cnt = w.len - n.s;
      if (o + cnt > cap) { err = 1; return o; }
      for (uint32_t q = w.lane; q < cnt; q += 32) {
        dst[o + q] = w.seq[n.s + q];
        if (kTrack) oout[o + q] = oin[n.s + q];
      }
      o += cnt;
    } else {
      if (o + 1 > cap) { err = 1; return o; }
      if (w.lane == 0) {
        dst[o] = (char)n.c;
        if (kTrack) oout[o] = GP_EDIT_INSERTED;
      }
      o++;
    }
  }
  __syncwarp();
  return o;
}

// Shared memory of one edit warp (dynamic: a CTA is kEditWarps warps, or kEditSmWarps when it owns its SM)
constexpr uint32_t kWarpSmemWords = 2u * (kInsZeroRow + 32u) + 2u * 5u * 32u + 192u + 32u;  // ins F/R, common chains, stage, seeds
constexpr uint32_t kWarpSmemBytes = kWarpSmemWords * 8u + kVBuf + 32u;                       // + stream ring + re-seed window
constexpr int kEditSmWarps = 12; // 12 x 32 x 168 registers: the whole register file of an SM

template<bool kTrack>
__global__ void __launch_bounds__(kEditSmWarps * 32, 1) edit_kernel(EditParams p)
{
  extern __shared__ __align__(16) uint64_t edit_dyn[];
  __shared__ unsigned char code_sh[256];
  for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) {
    const uint32_t lc = i | 0x20u;
    code_sh[i] = lc == 'a' ? 1 : lc == 'c' ? 2 : lc == 'g' ? 3 : lc == 't' ? 4 : 0;
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    atomicMin(p.counters + 4, t); // (several launches per pass: the first start)
  }
  unsigned long long n_trig = 0, n_edit = 0, n_mask = 0, n_roll = 0;
  for (;;) {
    uint32_t slot = 0;
    if (lane == 0) slot = atomicAdd(p.next_contig, 1u);
    slot = __shfl_sync(kFull, slot, 0);
    if (slot >= p.n_contigs) break;
    const uint32_t ci = p.order[slot];
    if (p.batch_done) { // pipelined with the filter build: wait until the contig's batch has its nk filters
      uint32_t ok = 1;
      if (lane == 0) {
        // acquire loads: the filter words read below (ld.global.cg, never the non-coherent path -- the build kernel
        // is writing the pool while this kernel runs) must not be satisfied before the flag has been seen
        const uint32_t* flag = p.batch_done + p.contig_batch[ci];
        const uint32_t* progress = p.batch_done + p.n_batches; // filters finished so far, all batches
        unsigned long long t0 = 0, t1 = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        uint32_t seen = ld_acquire_u32(progress), naps = 0;
        unsigned ns = 128;
        while (ld_acquire_u32(flag) < p.nk) {
          __nanosleep(ns);
          if (ns < 2048) ns <<= 1; // back off: hundreds of waiting warps must not hammer the two words they all read
          if ((++naps & 15u) == 0u) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            const uint32_t now = ld_acquire_u32(progress);
            if (now != seen) { seen = now; t0 = t1; }
            else if (t1 - t0 > 4000000000ull) { ok = 0; break; } // 4 s without ANY new filter: the build is not running beside us
          }
        }
        __threadfence();
      }
      ok = __shfl_sync(kFull, ok, 0);
      if (!ok) { if (lane == 0) atomicExch(p.error, 2); break; } // the host re-runs the polish after the build
    }
    const uint64_t off = p.cap_off[ci];
    const uint32_t cap = uint32_t(p.cap_off[ci + 1] - off);
    uint32_t len = p.cur_len[ci];
    uint32_t cur = 0;
    bool dropped = false;
    WS w;
    w.lane = lane;
    {
      uint64_t* base = edit_dyn + size_t(warp) * (kWarpSmemBytes / 8u);
      w.insF = base;
      w.insR = base + (kInsZeroRow + 32u);
      w.com = base + 2u * (kInsZeroRow + 32u);
      w.stage = w.com + 2u * 5u * 32u;
      w.seedt = w.stage + 192u;
      w.vb = reinterpret_cast<unsigned char*>(w.seedt + 32u);
      w.kmer = w.vb + kVBuf;
    }
    w.code = code_sh;
    w.nd = p.nodes + p.node_off[ci];
    w.ncap = uint32_t(p.node_off[ci + 1] - p.node_off[ci]);
    w.max_ins = p.max_insertions; w.max_del = p.max_deletions; w.jump = p.jump;
    w.mode = p.mode; w.mask = p.mask;
    w.err = 0;
    w.n_trig = w.n_edit = w.n_mask = w.n_roll = 0;
    for (uint32_t ki = 0; ki < p.nk; ki++) {
      if (len < p.min_contig_len) { dropped = true; break; } // readAndCorrect, :1850
      w.seq = p.buf[cur] + off;
      w.len = len;
      w.k = p.k[ki];
      w.icap = p.insertion_cap[ki];
      w.thrM = p.thr_missing[ki]; w.thrE = p.thr_edit[ki]; w.thrD = p.thr_del[ki];
      w.mul1 = 1ull ^ (uint64_t(w.k) * kMultiSeed);
      w.mul2 = 2ull ^ (uint64_t(w.k) * kMultiSeed);
      w.mul3 = 3ull ^ (uint64_t(w.k) * kMultiSeed);
      w.bf = p.bf_pool + (uint64_t(p.bf_slot ? p.bf_slot[p.contig_batch[ci]] : p.contig_batch[ci]) * p.nk + ki) * kBfWords;
      w.nn = 0;
      edit_round(w);
      __syncwarp();
      int err = w.err;
      const uint32_t nl = err ? 0u : emit_rope<kTrack>(w, p.buf[cur ^ 1u] + off, cap, err, kTrack ? p.orig[cur] + off : nullptr,
                                                       kTrack ? p.orig[cur ^ 1u] + off : nullptr);
      if (err) { if (lane == 0) atomicExch(p.error, 1); break; }
      __syncwarp();
      len = nl;
      cur ^= 1u;
    }
    if (lane == 0) {
      p.cur_len[ci] = len;
      p.which[ci] = (uint8_t)cur;
      p.dropped[ci] = dropped ? 1 : 0;
    }
    n_trig += w.n_trig; n_edit += w.n_edit; n_mask += w.n_mask; n_roll += w.n_roll;
  }
  if (lane == 0) {
    if (n_trig) atomicAdd(p.counters + 0, n_trig);
    if (n_edit) atomicAdd(p.counters + 1, n_edit);
    if (n_mask) atomicAdd(p.counters + 2, n_mask);
    if (n_roll) atomicAdd(p.counters + 3, n_roll);
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    atomicMax(p.counters + 5, t);
  }
}

// alongside_build (gp_pipeline_run): launched right behind the level-synchronous build kernel in the same
// stream with programmatic stream serialization -- it starts once every build CTA has signalled
// launch_dependents, i.e. when the build is resident.  Two shapes:
//   alongside_build = 1  one 3-warp CTA per SM beside 2 build CTAs (per scheduler: 2 x 2 build warps x 80 registers +
//                        one edit warp x 168 registers <= 16384): the two kernels share every SM;
//   alongside_build = 2  CTAs of kEditSmWarps warps, each the whole register file of an SM: they only fit on SMs that
//                        the build kernel has given back (LevelParams::reserve_sms) -- and, one per SM, everywhere
//                        once the build kernel is through, which is what takes the tail.
constexpr int kAlongsideWarps = 3;

// load the kernel now (lazy module loading would otherwise do it at the first launch -- and that launch would wait for
// everything already running, e.g. the build kernel it is meant to run beside)
void preload_edit()
{
  for (const void* f : { (const void*)edit_kernel<false>, (const void*)edit_kernel<true> }) {
    cudaFuncAttributes a;
    if (cudaFuncGetAttributes(&a, f) != cudaSuccess) cudaGetLastError();
    cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, kEditSmWarps * int(kWarpSmemBytes));
  }
}

cudaError_t launch_edit(const EditParams& p, int sm_count, cudaStream_t s, int alongside_build)
{
  if (p.n_contigs == 0) return cudaSuccess;
  void (*const kern)(EditParams) = p.orig[0] ? edit_kernel<true> : edit_kernel<false>;
  if (alongside_build && std::getenv("GP_EXP_NO_EDIT")) return cudaSuccess; // (experiment: what the build costs in this mode by itself)
  // (function attributes are per device: set on every launch, a cheap host-side call)
  cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kEditSmWarps * int(kWarpSmemBytes));
  // same shared-memory carve-out as the build kernel (132 KB), so that the two can share an SM; a CTA that owns its
  // SM asks for what it needs
  cudaFuncSetAttribute((const void*)kern, cudaFuncAttributePreferredSharedMemoryCarveout, alongside_build == 2 ? 72 : 58);
  if (alongside_build) {
    const uint32_t warps = alongside_build == 2 ? uint32_t(kEditSmWarps) : uint32_t(kAlongsideWarps);
    uint32_t grid = uint32_t(sm_count);
    const uint32_t need = (p.n_contigs + warps - 1) / warps;
    if (grid > need) grid = need;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(warps * 32);
    cfg.dynamicSmemBytes = warps * kWarpSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kern, p) == cudaSuccess) return cudaSuccess;
    cudaGetLastError(); // no programmatic launch on this driver: an ordinary launch runs after the build (correct, no overlap)
    kern<<<grid, warps * 32, warps * kWarpSmemBytes, s>>>(p);
    return cudaGetLastError();
  }
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kEditWarps * 32, kEditWarps * kWarpSmemBytes);
  if (per_sm < 1) per_sm = 1;
  uint32_t grid = uint32_t(sm_count) * uint32_t(per_sm);
  const uint32_t need = (p.n_contigs + kEditWarps - 1) / kEditWarps;
  if (grid > need) grid = need;
  kern<<<grid, kEditWarps * 32, kEditWarps * kWarpSmemBytes, s>>>(p);
  return cudaGetLastError();
}

} // namespace gp
