// Host side of the GoldPolish drop-ins: everything that decides WHICH bytes reach the GPU.
//
// New C++ written against the behaviour of bcgsc/goldpolish (cited per function):
//   SeqIndex      src/seqindex.cpp:12-142, src/seqindex.hpp:59-102
//   Mappings      src/mappings.cpp:15-330
//   selection     src/goldpolish_targeted_bfs.cpp:86-133
//   .bf container btllib::KmerBloomFilter::save / load (btllib is not in the reference tree:
//                 layout UNPINNED, kept in bf_format below and nowhere else)
//   FASTA reader  kseq.h semantics as used by subprojects/ntedit/ntedit.cpp:1829-1842
#pragma once

#include "../../include/goldpolish_b200.h"

#include <zlib.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <string_view>
#include <unordered_map>
#include <unordered_set>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

namespace gph {

[[noreturn]] inline void die(const std::string& msg)
{
  std::cerr << "[goldpolish_b200] [ERROR] " << msg << std::endl;
  std::exit(EXIT_FAILURE);
}
inline void info(const std::string& msg)
{
  if (!std::getenv("GP_QUIET")) std::cerr << "[goldpolish_b200] [INFO] " << msg << std::endl;
}
inline void check_gp(gp_ctx* ctx, int rc, const char* what)
{
  if (rc != GP_OK) die(std::string(what) + ": " + gp_last_error(ctx));
}
inline bool endswith(const std::string& s, const std::string& suf)
{
  return s.size() >= suf.size() && s.compare(s.size() - suf.size(), suf.size(), suf) == 0;
}

// ---------------------------------------------------------------------------------------
// Text files read by all host cores (SURVEY §8f rank 2): a read-only map of the file, cut at line ends into one slice
// per thread (at least 1 MiB of text each)
// ---------------------------------------------------------------------------------------
inline unsigned host_threads(unsigned threads)
{ // 0: GP_HOST_THREADS, else every core
  if (threads == 0)
    if (const char* e = std::getenv("GP_HOST_THREADS")) threads = unsigned(std::max(0, std::atoi(e)));
  return threads ? threads : std::max(1u, std::thread::hardware_concurrency());
}
inline bool is_space(char c) { return c == ' ' || (c >= '\t' && c <= '\r'); } // std::isspace in the "C" locale

struct SlicedFile {
  const char* d = nullptr;
  size_t N = 0, T = 1;
  std::vector<size_t> cut; // slice t = [cut[t], cut[t + 1]); every slice starts at a line start
  int fd = -1;
  bool mapped = false;
  std::string owned;       // decoded bytes of a compressed input

  // decode = true: a compressed or BAM file (by suffix) is decoded into memory first -- what btllib::DataSource does
  // for the reference's mapping files (src/mappings.cpp:136-139): .gz through zlib, .bz2 / .xz / .zst / .zip through
  // their tools, .bam through `samtools view -h`; a missing tool is an error, never a silently empty input
  SlicedFile(const std::string& path, unsigned threads, bool decode = false)
  {
    if (decode && decode_into(path, owned)) {
      d = owned.data();
      N = owned.size();
    } else {
      fd = open(path.c_str(), O_RDONLY);
      if (fd < 0) die("cannot open " + path);
      struct stat st;
      if (fstat(fd, &st) != 0) die("cannot stat " + path);
      N = size_t(st.st_size);
      if (N) {
        d = static_cast<const char*>(mmap(nullptr, N, PROT_READ, MAP_PRIVATE, fd, 0));
        if (d == MAP_FAILED) die("cannot map " + path);
        madvise(const_cast<char*>(d), N, MADV_SEQUENTIAL);
        mapped = true;
      }
    }
    T = std::max<size_t>(1, std::min<size_t>(host_threads(threads), N / (1u << 20) + 1));
    cut.assign(T + 1, N);
    cut[0] = 0;
    for (size_t t = 1; t < T; t++) {
      size_t pos = std::max(cut[t - 1], N / T * t);
      if (pos > 0 && pos < N && d[pos - 1] != '\n') {
        const char* q = static_cast<const char*>(memchr(d + pos, '\n', N - pos));
        pos = q ? size_t(q - d) + 1 : N;
      }
      cut[t] = std::min(pos, N);
    }
  }
  // false: a plain file (map it).  true: `out` holds the decoded bytes.
  static bool decode_into(const std::string& path, std::string& out)
  {
    if (endswith(path, ".gz")) {
      gzFile g = gzopen(path.c_str(), "rb");
      if (!g) die("cannot open " + path);
      gzbuffer(g, 1u << 20);
      std::vector<char> buf(4u << 20);
      for (;;) {
        const int n = gzread(g, buf.data(), unsigned(buf.size()));
        if (n < 0) die("cannot decompress " + path);
        if (n == 0) break;
        out.append(buf.data(), size_t(n));
      }
      gzclose(g);
      return true;
    }
    static const char* const tools[][2] = { { ".bam", "samtools view -h" }, { ".bz2", "bzip2 -dc" }, { ".xz", "xz -dc" },
                                            { ".zst", "zstd -dc" }, { ".zip", "unzip -p" }, { ".lrz", "lrzip -dqo -" } };
    for (const auto& t : tools) {
      if (!endswith(path, t[0])) continue;
      std::string quoted = "'";
      for (const char c : path) quoted += c == '\'' ? std::string("'\\''") : std::string(1, c);
      quoted += "'";
      const std::string cmd = std::string(t[1]) + " " + quoted;
      FILE* f = popen(cmd.c_str(), "r");
      if (!f) die("cannot run: " + cmd);
      std::vector<char> buf(4u << 20);
      size_t n;
      while ((n = std::fread(buf.data(), 1, buf.size(), f)) > 0) out.append(buf.data(), n);
      if (pclose(f) != 0) die("failed: " + cmd + " (is the tool installed?)");
      return true;
    }
    return false;
  }
  SlicedFile(const SlicedFile&) = delete;
  SlicedFile& operator=(const SlicedFile&) = delete;
  ~SlicedFile()
  {
    if (mapped) munmap(const_cast<char*>(d), N);
    if (fd >= 0) close(fd);
  }
  // fn(t) for every slice, one thread each
  template <class Fn> void parallel(Fn&& fn) const
  {
    std::vector<std::thread> th;
    for (size_t t = 1; t < T; t++) th.emplace_back(fn, t);
    fn(size_t(0));
    for (auto& x : th) x.join();
  }
  // whitespace-separated tokens of every slice (`stream >> token`), as views into the map.  Formats whose records are
  // `group` tokens whatever the line structure (the SeqIndex file: 4, ntLink mappings: 3) need every slice to hold
  // whole records: if one does not, all tokens are handed back as ONE slice
  std::vector<std::vector<std::string_view>> tokens(size_t group) const
  {
    std::vector<std::vector<std::string_view>> out(T);
    parallel([&](size_t t) {
      size_t pos = cut[t];
      const size_t end = cut[t + 1];
      auto& v = out[t];
      while (pos < end) {
        while (pos < end && is_space(d[pos])) pos++;
        const size_t b = pos;
        while (pos < end && !is_space(d[pos])) pos++;
        if (pos > b) v.emplace_back(d + b, pos - b);
      }
    });
    bool whole = true;
    for (const auto& v : out) whole = whole && v.size() % group == 0;
    if (!whole)
      for (size_t t = 1; t < T; t++) {
        out[0].insert(out[0].end(), out[t].begin(), out[t].end());
        std::vector<std::string_view>().swap(out[t]);
      }
    return out;
  }
};

// ---------------------------------------------------------------------------------------
// SeqIndex: id -> (byte offset of the sequence line, length, average phred)
// ---------------------------------------------------------------------------------------
struct SeqRecord {
  uint64_t start = 0, len = 0;
  double phred = 0.0;
};

class SeqIndex {
public:
  // Build from a FASTA with exactly 2 lines per record or a FASTQ with exactly 4
  // (src/seqindex.cpp:12-66).  The first duplicate id wins (unordered_map::emplace).
  // Same line arithmetic as the reference's getline loop (line i has phase i % 2 or i % 4, whatever it holds;
  // a '\r' stays part of its line), but over an mmap of the file with `threads` workers (SURVEY §8f rank 2):
  // every worker counts the newlines of its slice, a prefix sum gives the line number at every slice start, and
  // the worker then parses the records that START in its slice.  threads = 0: GP_INDEX_THREADS or all cores.
  static SeqIndex build(const std::string& seqs_path, unsigned threads = 0)
  {
    SeqIndex ix;
    ix.seqs_path = seqs_path;
    const int fd = open(seqs_path.c_str(), O_RDONLY);
    if (fd < 0) die("cannot open " + seqs_path);
    struct stat st;
    if (fstat(fd, &st) != 0) die("cannot stat " + seqs_path);
    const size_t N = size_t(st.st_size);
    if (N == 0) { close(fd); return ix; }
    const char* d = static_cast<const char*>(mmap(nullptr, N, PROT_READ, MAP_PRIVATE, fd, 0));
    if (d == MAP_FAILED) die("cannot map " + seqs_path);
    madvise(const_cast<char*>(d), N, MADV_SEQUENTIAL);
    const bool fastq = d[0] == '@';
    const size_t lpr = fastq ? 4 : 2;
    if (threads == 0) {
      if (const char* e = std::getenv("GP_INDEX_THREADS")) threads = unsigned(std::atoi(e));
      if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());
    }
    const size_t T = std::max<size_t>(1, std::min<size_t>(threads, N / (1u << 20) + 1));
    std::vector<size_t> cut(T + 1), nl(T + 1, 0);
    for (size_t t = 0; t <= T; t++) cut[t] = N / T * t;
    cut[T] = N;
    auto parallel = [&](auto&& fn) {
      std::vector<std::thread> th;
      for (size_t t = 1; t < T; t++) th.emplace_back(fn, t);
      fn(size_t(0));
      for (auto& x : th) x.join();
    };
    parallel([&](size_t t) { // newlines per slice
      size_t c = 0;
      const char* p = d + cut[t];
      const char* e = d + cut[t + 1];
      while (p < e) {
        p = static_cast<const char*>(memchr(p, '\n', size_t(e - p)));
        if (!p) break;
        c++; p++;
      }
      nl[t + 1] = c;
    });
    for (size_t t = 0; t < T; t++) nl[t + 1] += nl[t]; // newlines before slice t
    struct Rec { std::string id; uint64_t start, len; double phred; };
    std::vector<std::vector<Rec>> out(T);
    parallel([&](size_t t) {
      // first line that starts inside the slice, and its number
      size_t pos = cut[t], line = nl[t];
      if (pos != 0 && d[pos - 1] != '\n') {
        const char* q = static_cast<const char*>(memchr(d + pos, '\n', N - pos));
        if (!q) return;            // the slice is the middle of the last line
        pos = size_t(q - d) + 1;
        line++;
      }
      // skip to the first header line (phase 0)
      while (pos < N && line % lpr != 0) {
        const char* q = static_cast<const char*>(memchr(d + pos, '\n', N - pos));
        if (!q) return;
        pos = size_t(q - d) + 1;
        line++;
      }
      auto line_end = [&](size_t a) { // one past the last character of the line starting at a
        const char* q = a < N ? static_cast<const char*>(memchr(d + a, '\n', N - a)) : nullptr;
        return q ? size_t(q - d) : N;
      };
      while (pos < N && pos < cut[t + 1]) { // records that start in this slice
        Rec r;
        const size_t he = line_end(pos);
        {
          const char* sp = static_cast<const char*>(memchr(d + pos, ' ', he - pos));
          size_t ie = sp ? size_t(sp - d) : he;                 // split(line, " ")[0]
          size_t ib = ie > pos ? pos + 1 : pos;                 // without its first character
          if (fastq) {                                          // :33 cut at the first tab
            const char* tb = ib < ie ? static_cast<const char*>(memchr(d + ib, '\t', ie - ib)) : nullptr;
            if (tb) ie = size_t(tb - d);
          }
          r.id.assign(d + ib, ie - ib);
        }
        if (he >= N) break; // header without a sequence line: getline ends, nothing is recorded
        const size_t sb = he + 1;
        if (sb >= N) break;  // (an empty last line does not exist for getline)
        const size_t se = line_end(sb);
        r.start = sb; r.len = se - sb; r.phred = 0.0;
        size_t next = se + 1;
        if (!fastq) { out[t].push_back(std::move(r)); pos = next; continue; }
        // '+' line, then the quality line
        if (se >= N || next >= N) break;
        const size_t pe = line_end(next);
        if (pe >= N || pe + 1 >= N) break;
        const size_t qb = pe + 1, qe = line_end(qb);
        // calc_phred_avg(line, 0, line.size() - 1): the last quality character is left out (:45); btllib reads a
        // length of 0 as "the whole string" (a 1-character line is averaged over that character) and refuses a
        // range beyond the string (an empty line: size() - 1 wraps)
        if (qe == qb) die("calc_phred_avg: range exceeds string.");
        const size_t n = qe - qb > 1 ? qe - qb - 1 : 1;
        {
          size_t sum = 0;
          const unsigned char* qp = reinterpret_cast<const unsigned char*>(d + qb);
          for (size_t i = 0; i < n; i++) sum += qp[i];
          r.phred = double(sum) / double(n) - 33.0;
        }
        out[t].push_back(std::move(r));
        pos = qe + 1;
      }
    });
    size_t total = 0;
    for (auto& v : out) total += v.size();
    ix.shards[0].reserve(total);
    ix.order.reserve(total);
    for (auto& v : out)
      for (auto& r : v) ix.add(r.id, r.start, r.len, r.phred);
    munmap(const_cast<char*>(d), N);
    close(fd);
    return ix;
  }

  // id \t start \t len \t phred, default ostream formatting (src/seqindex.cpp:68-84)
  void save(const std::string& path) const
  {
    std::ofstream o(path);
    for (const auto& id : order) {
      const SeqRecord& r = at(id);
      o << id << '\t' << r.start << '\t' << r.len << '\t' << r.phred << '\n';
    }
  }

  // whitespace separated tokens, four per record (src/seqindex.cpp:86-125); the first duplicate id wins.  Loaded by
  // all host cores: tokens per slice of the file, then the ids are dealt to the threads by hash and every thread fills
  // its own shard of the map, walking the records in file order
  static SeqIndex load(const std::string& index_path, const std::string& seqs_path, unsigned threads = 0)
  {
    SeqIndex ix;
    ix.seqs_path = seqs_path;
    const SlicedFile f(index_path, threads);
    const auto toks = f.tokens(4);
    const size_t T = f.T;
    struct Rec { std::string_view id; uint64_t start, len; double phred; };
    std::vector<std::vector<Rec>> recs(T);
    std::vector<std::vector<uint8_t>> first(T);
    f.parallel([&](size_t t) {
      const auto& v = toks[t];
      recs[t].reserve(v.size() / 4);
      for (size_t i = 0; i + 3 < v.size(); i += 4) // (a trailing partial record never reaches the fourth token)
        recs[t].push_back(Rec{ v[i], to_u64(v[i + 1]), to_u64(v[i + 2]), to_double(v[i + 3]) });
      first[t].assign(recs[t].size(), 0);
    });
    ix.shards.assign(T, Shard());
    f.parallel([&](size_t me) {
      Shard& mine = ix.shards[me];
      const std::hash<std::string_view> H;
      for (size_t t = 0; t < T; t++)
        for (size_t i = 0; i < recs[t].size(); i++) {
          const Rec& r = recs[t][i];
          if (T > 1 && H(r.id) % T != me) continue;
          SeqRecord sr;
          sr.start = r.start; sr.len = r.len; sr.phred = r.phred;
          if (mine.emplace(std::string(r.id), sr).second) first[t][i] = 1;
        }
    });
    std::vector<std::vector<std::string>> ord(T);
    f.parallel([&](size_t t) {
      for (size_t i = 0; i < recs[t].size(); i++)
        if (first[t][i]) ord[t].emplace_back(recs[t][i].id);
    });
    size_t total = 0;
    for (const auto& v : ord) total += v.size();
    ix.order.reserve(total);
    for (auto& v : ord)
      for (auto& id : v) ix.order.push_back(std::move(id));
    return ix;
  }

  bool exists(const std::string& id) const { return find(id) != nullptr; }
  const SeqRecord& at(const std::string& id) const
  {
    const SeqRecord* r = find(id);
    if (!r) die("sequence id not in index: " + id); // unordered_map::at would throw
    return *r;
  }
  size_t size() const
  {
    size_t n = 0;
    for (const Shard& m : shards) n += m.size();
    return n;
  }

  // whole sequence line, as SeqIndex::get_seq<1> returns it (src/seqindex.hpp:59-102)
  void read_seq(const std::string& id, std::string& out) const
  {
    const SeqRecord& r = at(id);
    if (r.len >= 20ull * 1024ull * 1024ull) die("Seq size over buffer size."); // :88-90
    if (fd < 0) {
      fd = open(seqs_path.c_str(), O_RDONLY);
      if (fd < 0) die("cannot open " + seqs_path);
    }
    out.resize(r.len);
    size_t got = 0;
    while (got < r.len) {
      const ssize_t n = pread(fd, &out[got], r.len - got, off_t(r.start + got));
      if (n <= 0) die("read did not read all bytes.");
      got += size_t(n);
    }
  }

  // The sequences of ids[first .. first + n) back to back in `out` (the slab the server hands to gp_reads_append), read
  // by `threads` workers: the offsets follow from the index, every worker preads its share of the reads into place.
  void read_many(const std::vector<const std::string*>& ids, size_t first, size_t n, std::string& out, unsigned threads = 0) const
  {
    std::vector<const SeqRecord*> recs(n);
    std::vector<size_t> off(n + 1, 0);
    for (size_t i = 0; i < n; i++) {
      recs[i] = &at(*ids[first + i]);
      if (recs[i]->len >= 20ull * 1024ull * 1024ull) die("Seq size over buffer size."); // :88-90
      off[i + 1] = off[i] + recs[i]->len;
    }
    out.resize(off[n]);
    if (fd < 0) {
      fd = open(seqs_path.c_str(), O_RDONLY);
      if (fd < 0) die("cannot open " + seqs_path);
    }
    const size_t T = std::max<size_t>(1, std::min<size_t>(host_threads(threads), off[n] / (4u << 20) + 1));
    auto work = [&](size_t t) { // reads whose first byte falls into the t-th part of the slab
      const size_t lo = off[n] / T * t, hi = t + 1 == T ? off[n] + 1 : off[n] / T * (t + 1);
      for (size_t i = size_t(std::lower_bound(off.begin(), off.begin() + n, lo) - off.begin()); i < n && off[i] < hi; i++) {
        size_t got = 0;
        while (got < recs[i]->len) {
          const ssize_t r = pread(fd, &out[off[i] + got], recs[i]->len - got, off_t(recs[i]->start + got));
          if (r <= 0) die("read did not read all bytes.");
          got += size_t(r);
        }
      }
    };
    std::vector<std::thread> th;
    for (size_t t = 1; t < T; t++) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
  }

  std::string seqs_path;
  std::vector<std::string> order; // insertion order (save() of the reference iterates a hash map)

private:
  using Shard = std::unordered_map<std::string, SeqRecord>;
  const SeqRecord* find(const std::string& id) const
  {
    const Shard& m = shards[shards.size() > 1 ? std::hash<std::string>{}(id) % shards.size() : 0];
    const auto it = m.find(id);
    return it == m.end() ? nullptr : &it->second;
  }
  void add(const std::string& id, uint64_t start, uint64_t len, double phred)
  {
    Shard& m = shards[shards.size() > 1 ? std::hash<std::string>{}(id) % shards.size() : 0];
    if (m.find(id) != m.end()) return;
    SeqRecord r;
    r.start = start; r.len = len; r.phred = phred;
    m.emplace(id, r);
    order.push_back(id);
  }
  // std::stoull / std::stod of the reference (:105-113); plain digit strings take the short way
  static uint64_t to_u64(std::string_view t)
  {
    uint64_t v = 0;
    bool plain = !t.empty() && t.size() < 19;
    for (const char c : t) {
      if (c < '0' || c > '9') { plain = false; break; }
      v = v * 10 + unsigned(c - '0');
    }
    if (plain) return v;
    try {
      return std::stoull(std::string(t));
    } catch (const std::exception&) {
      die("index: '" + std::string(t) + "' is not a number");
    }
  }
  static double to_double(std::string_view t)
  {
    try {
      return std::stod(std::string(t));
    } catch (const std::exception&) {
      die("index: '" + std::string(t) + "' is not a number");
    }
  }
  std::vector<Shard> shards = std::vector<Shard>(1); // an id lives in shard hash(id) % shards.size()
  mutable int fd = -1;
};

// ---------------------------------------------------------------------------------------
// Mappings: target id -> mapped read ids, first-seen order, de-duplicated
// ---------------------------------------------------------------------------------------
// Same result as AllMappings (src/mappings.cpp:15-330), loaded by all host cores (SURVEY §8f rank 2) instead of one
// stream-parsing thread:
//   1. the file is mapped and cut at line ends into one slice per thread (SlicedFile); every thread tokenises its slice
//      into (read, target, minimizers) records that point into the map (no copies);
//   2. the reference's carry-over -- a line with too few columns keeps the ids of the line before it (:146-160,
//      :199-213), ntLink tokens are triples whatever the line structure (:83-108) -- is resolved by one short sequential
//      pass over the slices that need it (none, in a well-formed file);
//   3. targets are dealt to the threads by hash; every thread walks ALL records in file order and keeps those of its
//      own targets, so "first seen" is the file's order and no map is shared; it then applies the minimizer filter
//      (:230-320) to its targets and turns the survivors into strings.
// threads = 0: GP_HOST_THREADS or all cores.
class Mappings {
public:
  using Map = std::unordered_map<std::string, std::vector<std::string>>;

  // src/mappings.cpp:15-35: type by file suffix; the minimizer filter only for ntLink triples
  Mappings(const std::string& path, const SeqIndex& targets, unsigned mx_min, unsigned mx_max, double mx_max_per_10kbp,
           unsigned threads = 0)
  {
    // (.bam reads as SAM through samtools, as btllib::DataSource pipes it; any other suffix -- "x.paf.gz" included,
    // as in the reference -- is ntLink triples; compressed files are decoded first, see SlicedFile)
    const int target_col = endswith(path, ".sam") || endswith(path, ".bam") ? 3 : endswith(path, ".paf") ? 6 : 0;
    if (target_col == 0) {
      if (mx_max_per_10kbp <= 0) die("max_mapped_seqs_per_target_10kbp is not positive.");
      if (mx_min >= mx_max) die("mx_threshold_min is not smaller than mx_threshold_max.");
    }
    load(path, targets, target_col, mx_min, mx_max, mx_max_per_10kbp, threads);
  }

  const std::vector<std::string>& get(const std::string& target) const
  {
    static const std::vector<std::string> empty;
    const Map& m = shards[std::hash<std::string>{}(target) % shards.size()];
    const auto it = m.find(target);
    return it == m.end() ? empty : it->second;
  }
  // every (target, reads) pair, in no particular order
  template <class Fn> void for_each(Fn&& fn) const
  {
    for (const Map& m : shards)
      for (const auto& kv : m) fn(kv.first, kv.second);
  }
  size_t n_targets() const
  {
    size_t n = 0;
    for (const Map& m : shards) n += m.size();
    return n;
  }

private:
  using sv = std::string_view;
  struct Rec {
    sv read, target;
    unsigned long mx = 0;
    bool has_read = false, has_target = false;
  };
  struct Slice {
    std::vector<Rec> recs;
    bool incomplete = false;   // some record lacks an id of its own
  };
  static unsigned long parse_mx(sv t)
  { // std::stoul (:95); digits-only tokens take the short way
    unsigned long v = 0;
    bool plain = !t.empty() && t.size() < 19;
    for (const char c : t) {
      if (c < '0' || c > '9') { plain = false; break; }
      v = v * 10 + unsigned(c - '0');
    }
    if (plain) return v;
    try {
      return std::stoul(std::string(t));
    } catch (const std::exception&) {
      die("mappings: '" + std::string(t) + "' is not a minimizer count"); // (the reference dies of the uncaught exception)
    }
  }
  static unsigned count_ge(const std::vector<unsigned>& v, unsigned thr)
  {
    unsigned c = 0;
    for (const auto x : v) c += x >= thr ? 1u : 0u;
    return c;
  }

  void load(const std::string& path, const SeqIndex& targets, int target_col, unsigned mx_min, unsigned mx_max,
            double max_per_10kbp, unsigned threads)
  {
    const SlicedFile f(path, threads, true);
    const char* d = f.d;
    const size_t T = f.T;
    shards.assign(T, Map());
    auto parallel = [&](auto&& fn) { f.parallel(fn); };
    // 1. + 2. records per slice, carry-over resolved
    std::vector<Slice> sl(T);
    if (target_col == 0) {
      const auto toks = f.tokens(3);
      parallel([&](size_t t) {
        const auto& v = toks[t];
        sl[t].recs.reserve(v.size() / 3);
        for (size_t i = 0; i + 2 < v.size(); i += 3) { // (a trailing partial triple never reaches `case 2`)
          Rec r;
          r.read = v[i]; r.target = v[i + 1]; r.has_read = r.has_target = true;
          r.mx = parse_mx(v[i + 2]);
          if (r.mx >= mx_min) sl[t].recs.push_back(r); // :96
        }
      });
    } else {
      parallel([&](size_t t) {
        Slice& S = sl[t];
        size_t pos = f.cut[t];
        const size_t end = f.cut[t + 1];
        while (pos < end) { // one record per line that does not start with '@'
          const char* q = static_cast<const char*>(memchr(d + pos, '\n', end - pos));
          const size_t le = q ? size_t(q - d) : end;
          if (d[pos] != '@') {
            Rec r;
            int col = 1;
            size_t p = pos;
            while (p < le && col <= target_col) {
              while (p < le && is_space(d[p])) p++;
              const size_t b = p;
              while (p < le && !is_space(d[p])) p++;
              if (p == b) break;
              if (col == 1) { r.read = sv(d + b, p - b); r.has_read = true; }
              else if (col == target_col) { r.target = sv(d + b, p - b); r.has_target = true; }
              col++;
            }
            if (!r.has_read || !r.has_target) S.incomplete = true;
            S.recs.push_back(r);
          }
          pos = le + 1;
        }
      });
      sv read, target; // ids of the line before (empty strings before the first line, :144, :197)
      for (Slice& S : sl) {
        if (S.incomplete)
          for (Rec& r : S.recs) {
            if (!r.has_read) r.read = read;
            if (!r.has_target) r.target = target;
            read = r.read; target = r.target;
          }
        else if (!S.recs.empty()) { read = S.recs.back().read; target = S.recs.back().target; }
      }
    }
    // 3. one shard of targets per thread
    parallel([&](size_t me) {
      struct Entry {
        bool known = false;
        std::vector<sv> reads;
        std::unordered_set<sv> seen;
        std::vector<unsigned> mx;
      };
      std::unordered_map<sv, Entry> mine;
      const std::hash<sv> H;
      for (const Slice& S : sl)
        for (const Rec& r : S.recs) {
          if (T > 1 && H(r.target) % T != me) continue;
          auto it = mine.find(r.target);
          if (it == mine.end()) { // load_mapping, :37-72: targets that the index does not know are ignored
            it = mine.emplace(r.target, Entry()).first;
            it->second.known = targets.exists(std::string(r.target));
          }
          Entry& e = it->second;
          if (!e.known || !e.seen.insert(r.read).second) continue;
          e.reads.push_back(r.read);
          e.mx.push_back(unsigned(r.mx));
        }
      Map& out = shards[me];
      for (auto& kv : mine) {
        Entry& e = kv.second;
        if (!e.known || e.reads.empty()) continue;
        int thr = 0;
        if (target_col == 0) { // filter, :230-320
          const int max_reads = int(std::ceil(double(targets.at(std::string(kv.first)).len) * max_per_10kbp / 10000.0));
          if (max_reads <= 0) die("max_mapped_seqs <= 0.");
          int lo = int(mx_min), hi = int(mx_max);
          if (int(e.reads.size()) <= max_reads) thr = lo;
          else if (int(count_ge(e.mx, unsigned(hi))) > max_reads) thr = hi;
          else {
            while (hi - lo > 1) {
              const int mid = (hi + lo) / 2;
              if (int(count_ge(e.mx, unsigned(mid))) > max_reads) lo = mid; else hi = mid;
            }
            thr = hi;
          }
        }
        std::vector<std::string>& kept = out[std::string(kv.first)];
        for (size_t i = 0; i < e.reads.size(); i++)
          if (target_col != 0 || int(e.mx[i]) >= thr) kept.emplace_back(e.reads[i]);
      }
    });
  }

  std::vector<Map> shards; // target -> reads; a target lives in shard hash(target) % shards.size()
};

// ---------------------------------------------------------------------------------------
// read selection for one target (src/goldpolish_targeted_bfs.cpp:95-125)
// ---------------------------------------------------------------------------------------
struct Selection {
  std::vector<std::string> reads; // in fill order
  int kmer_threshold = 0;
};

inline Selection select_reads(const std::vector<std::string>& mapped, const SeqIndex& reads_index, uint64_t target_len,
                              double subsample_max_per_10kbp)
{
  Selection sel;
  const size_t n_adj = std::min<size_t>(mapped.size(), size_t(gp_mappings_cap(target_len, subsample_max_per_10kbp)));
  std::vector<std::pair<std::string, size_t>> v;
  v.reserve(mapped.size());
  for (const auto& id : mapped) v.emplace_back(id, size_t(reads_index.at(id).phred)); // tuple<SeqId, size_t>
  std::sort(v.begin(), v.end(), [](const auto& a, const auto& b) {
    return (a.second > b.second) || (a.second == b.second && a.first < b.first);
  });
  uint64_t bases = 0;
  for (size_t i = 0; i < n_adj; i++) bases += reads_index.at(v[i].first).len;
  sel.kmer_threshold = gp_kmer_threshold(bases);
  if (sel.kmer_threshold <= 0) die("k-mer threshold must be >0.");
  for (size_t i = 0; i < n_adj; i++) sel.reads.push_back(v[i].first);
  return sel;
}

// ---------------------------------------------------------------------------------------
// .bf container (btllib KmerBloomFilter).  UNPINNED: see file header.
// ---------------------------------------------------------------------------------------
namespace bf_format {

inline const char* signature()
{
  const char* s = std::getenv("GP_BF_SIGNATURE");
  return s ? s : "[BTLKmerBloomFilter_v6]";
}
inline const char* hash_fn()
{
  const char* s = std::getenv("GP_BF_HASH_FN");
  return s ? s : "ntHash_v2";
}
constexpr unsigned kPlaceholderNewlines = 50;

inline void save(const std::string& path, const uint8_t* payload, size_t bytes, unsigned hash_num, unsigned k)
{
  std::ofstream o(path, std::ios::out | std::ios::binary);
  if (!o.good()) die("cannot write " + path);
  o << signature() << '\n'
    << "bytes = " << bytes << '\n'
    << "hash_fn = \"" << hash_fn() << "\"\n"
    << "hash_num = " << hash_num << '\n'
    << "k = " << k << '\n'
    << "[HeaderEnd]\n";
  for (unsigned i = 0; i < kPlaceholderNewlines; i++) {
    if (i == 1) o << "  <binary data>";
    o << '\n';
  }
  o.write(reinterpret_cast<const char*>(payload), std::streamsize(bytes));
}

struct Header {
  size_t bytes = 0;
  unsigned hash_num = 0, k = 0;
};

// Reads any "[BTLKmerBloomFilter_v*]" header; the payload is the LAST `bytes` bytes of the file,
// which is robust to the number of placeholder lines a given btllib version writes.
inline Header load(const std::string& path, std::vector<uint8_t>& payload)
{
  std::ifstream f(path, std::ios::in | std::ios::binary);
  if (!f.good()) die("cannot open " + path);
  Header h;
  std::string line;
  bool sig = false, end = false;
  while (bool(std::getline(f, line))) {
    if (line == "[HeaderEnd]") { end = true; break; }
    if (!sig) {
      if (line.rfind("[BTLKmerBloomFilter_v", 0) != 0) die("Bloom filter file supplied (-r) is incorrect: " + path);
      sig = true;
      continue;
    }
    const auto eq = line.find('=');
    if (eq == std::string::npos) continue;
    auto trim = [](std::string s) {
      const auto b = s.find_first_not_of(" \t\"");
      const auto e = s.find_last_not_of(" \t\"\r");
      return b == std::string::npos ? std::string() : s.substr(b, e - b + 1);
    };
    const auto key = trim(line.substr(0, eq)), val = trim(line.substr(eq + 1));
    if (key == "bytes") h.bytes = std::stoull(val);
    else if (key == "hash_num") h.hash_num = unsigned(std::stoul(val));
    else if (key == "k") h.k = unsigned(std::stoul(val));
  }
  if (!end || h.bytes == 0) die("Bloom filter file supplied (-r) is incorrect: " + path);
  f.seekg(0, std::ios::end);
  const auto size = size_t(f.tellg());
  if (size < h.bytes) die("truncated Bloom filter payload: " + path);
  payload.resize(h.bytes);
  f.seekg(std::streamoff(size - h.bytes), std::ios::beg);
  f.read(reinterpret_cast<char*>(payload.data()), std::streamsize(h.bytes));
  return h;
}

} // namespace bf_format

// ---------------------------------------------------------------------------------------
// flagged-region BED: the lower-case runs that ntEdit -a1 leaves (ntedit.cpp:1131-1146), one row per run
// ---------------------------------------------------------------------------------------
inline void write_flagged_bed(const std::string& path, const std::vector<std::string>& names, const char* seqs,
                              const std::vector<uint64_t>& offsets)
{
  const uint32_t n = uint32_t(names.size());
  uint64_t cap = 4096;
  std::vector<uint32_t> rec;
  std::vector<uint64_t> st, en;
  uint64_t got;
  for (;;) {
    rec.resize(cap); st.resize(cap); en.resize(cap);
    got = gp_flagged_bed(seqs, offsets.data(), n, rec.data(), st.data(), en.data(), cap);
    if (got <= cap) break;
    cap = got;
  }
  std::ofstream o(path);
  if (!o.good()) die("cannot write " + path);
  for (uint64_t i = 0; i < got; i++) o << names[rec[i]] << '\t' << st[i] << '\t' << en[i] << '\n';
}

// ---------------------------------------------------------------------------------------
// edit records (gp_polish_fetch_edits) as VCF 4.2: one ##contig line per input record, records in input order then POS
// ---------------------------------------------------------------------------------------
struct EditRecords {
  std::vector<uint64_t> offsets; // n_contigs + 1
  std::vector<gp_edit> edits;
  std::vector<char> alleles;
};

inline EditRecords fetch_edits(gp_ctx* ctx, uint32_t n_contigs)
{
  EditRecords r;
  r.offsets.assign(size_t(n_contigs) + 1, 0);
  uint64_t need[2] = { 0, 0 };
  int rc = gp_polish_fetch_edits(ctx, r.offsets.data(), nullptr, 0, nullptr, 0, need);
  if (rc == GP_ERR_ARG && (need[0] || need[1])) {
    r.edits.resize(need[0]);
    r.alleles.resize(need[1]);
    rc = gp_polish_fetch_edits(ctx, r.offsets.data(), r.edits.data(), need[0], r.alleles.data(), need[1], need);
  }
  check_gp(ctx, rc, "gp_polish_fetch_edits");
  return r;
}

// names: CHROM of each input record (its name up to the first whitespace); lengths: draft lengths.  recs == nullptr
// writes the header only.
inline void write_edits_vcf(const std::string& path, const std::vector<std::string>& names, const std::vector<uint64_t>& lengths,
                            const EditRecords* recs)
{
  static const char* const kType[] = { "SNV", "MNV", "INS", "DEL", "COMPLEX" };
  std::ofstream o(path);
  if (!o.good()) die("cannot write " + path);
  o << "##fileformat=VCFv4.2\n##source=goldpolish_b200\n";
  for (size_t c = 0; c < names.size(); c++) o << "##contig=<ID=" << names[c] << ",length=" << lengths[c] << ">\n";
  o << "##INFO=<ID=TYPE,Number=1,Type=String,Description=\"Edit made by polishing: SNV, MNV, INS, DEL or COMPLEX\">\n";
  o << "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n";
  if (!recs) return;
  for (size_t c = 0; c < names.size(); c++)
    for (uint64_t r = recs->offsets[c]; r < recs->offsets[c + 1]; r++) {
      const gp_edit& e = recs->edits[r];
      const char* a = recs->alleles.data() + e.allele_off;
      o << names[c] << '\t' << uint64_t(e.pos) + 1 << "\t.\t";
      o.write(a, e.ref_len);
      o << '\t';
      o.write(a + e.ref_len, e.alt_len);
      o << "\t.\tPASS\tTYPE=" << (e.type < 5 ? kType[e.type] : "COMPLEX") << '\n';
    }
  if (!o.good()) die("cannot write " + path);
}

// ---------------------------------------------------------------------------------------
// k-mer support (gp_polish_fetch_support) as a TSV of k-mer completeness and Merqury's QV, per input record and k
// ---------------------------------------------------------------------------------------
struct KmerSupport {
  std::vector<gp_kmer_support> counts; // n_contigs * nk, contig-major
  std::vector<uint64_t> bits;          // n_batches * nk, batch-major
};

inline KmerSupport fetch_support(gp_ctx* ctx, uint32_t n_contigs, uint32_t nk, uint32_t n_batches)
{
  KmerSupport s;
  s.counts.resize(std::max<size_t>(size_t(n_contigs) * nk, 1));
  s.bits.resize(std::max<size_t>(size_t(n_batches) * nk, 1));
  check_gp(ctx, gp_polish_fetch_support(ctx, s.counts.data(), s.bits.data()), "gp_polish_fetch_support");
  s.counts.resize(size_t(n_contigs) * nk);
  s.bits.resize(size_t(n_batches) * nk);
  return s;
}

// E = 1 - (1 - missing / kmers)^(1/k), QV = -10 log10(E): "inf" without a missing k-mer, "NA" without a k-mer
inline std::string kmer_qv(uint64_t kmers, uint64_t missing, uint32_t k)
{
  if (kmers == 0) return "NA";
  if (missing == 0) return "inf";
  const double e = 1.0 - std::pow(1.0 - double(missing) / double(kmers), 1.0 / double(k));
  char b[64];
  std::snprintf(b, sizeof b, "%.4f", -10.0 * std::log10(e) + 0.0); // (+ 0.0: QV 0 prints without a sign)
  return b;
}

// names: one per input record, in the order of the counts; polished_is_draft: the 0.75 guard kept the input, so the
// polished columns describe the draft
inline void write_kmer_qv(const std::string& path, const std::vector<std::string>& names, const std::vector<uint32_t>& ks,
                          const KmerSupport& s, bool polished_is_draft)
{
  const size_t nk = ks.size(), nb = nk ? s.bits.size() / nk : 0;
  std::ofstream o(path);
  if (!o.good()) die("cannot write " + path);
  char b[64];
  o << "#goldpolish_b200 k-mer support: k-mers per record position, missing = not contained in the filter of its batch\n#k";
  for (uint32_t k : ks) o << '\t' << k;
  o << "\n#filter_fill";
  for (size_t j = 0; j < nk; j++) { // set bits over all batches' filters of this k
    uint64_t set = 0;
    for (size_t bt = 0; bt < nb; bt++) set += s.bits[bt * nk + j];
    if (nb) std::snprintf(b, sizeof b, "%.6f", double(set) / (double(nb) * 4194304.0));
    o << '\t' << (nb ? b : "NA");
  }
  o << "\n#filter_fp_rate";
  for (size_t j = 0; j < nk; j++) { // (set / 2^22)^4, the mean over the batches
    double fp = 0;
    for (size_t bt = 0; bt < nb; bt++) fp += std::pow(double(s.bits[bt * nk + j]) / 4194304.0, 4.0);
    if (nb) std::snprintf(b, sizeof b, "%.6g", fp / double(nb));
    o << '\t' << (nb ? b : "NA");
  }
  o << "\n#name\tk\tdraft_kmers\tdraft_missing\tdraft_qv\tpolished_kmers\tpolished_missing\tpolished_qv\n";
  std::vector<uint64_t> tot(4 * nk, 0);
  for (size_t c = 0; c < names.size(); c++)
    for (size_t j = 0; j < nk; j++) {
      const gp_kmer_support& e = s.counts[c * nk + j];
      const uint64_t dk = e.draft_kmers, dm = e.draft_kmers - e.draft_present;
      const uint64_t pk = polished_is_draft ? dk : e.polished_kmers;
      const uint64_t pm = polished_is_draft ? dm : e.polished_kmers - e.polished_present;
      o << names[c] << '\t' << ks[j] << '\t' << dk << '\t' << dm << '\t' << kmer_qv(dk, dm, ks[j]) << '\t' << pk << '\t' << pm
        << '\t' << kmer_qv(pk, pm, ks[j]) << '\n';
      tot[4 * j] += dk; tot[4 * j + 1] += dm; tot[4 * j + 2] += pk; tot[4 * j + 3] += pm;
    }
  for (size_t j = 0; j < nk; j++)
    o << "*\t" << ks[j] << '\t' << tot[4 * j] << '\t' << tot[4 * j + 1] << '\t' << kmer_qv(tot[4 * j], tot[4 * j + 1], ks[j]) << '\t'
      << tot[4 * j + 2] << '\t' << tot[4 * j + 3] << '\t' << kmer_qv(tot[4 * j + 2], tot[4 * j + 3], ks[j]) << '\n';
  if (!o.good()) die("cannot write " + path);
}

// ---------------------------------------------------------------------------------------
// runs of unsupported k-mers (gp_polish_fetch_unsupported) as BED rows
// ---------------------------------------------------------------------------------------
struct UnsupportedRuns {
  std::vector<uint64_t> off;             // n_contigs * 2 * nk + 1: runs of (c, r, j) at off[(c * 2 + r) * nk + j] ..
  std::vector<gp_unsupported_run> runs;
};

inline UnsupportedRuns fetch_unsupported(gp_ctx* ctx, uint32_t n_contigs, uint32_t nk)
{
  UnsupportedRuns u;
  u.off.resize(size_t(n_contigs) * 2 * nk + 1);
  uint64_t needed = 0;
  int rc = gp_polish_fetch_unsupported(ctx, u.off.data(), nullptr, 0, &needed);
  if (rc == GP_ERR_ARG && needed) {
    u.runs.resize(needed);
    rc = gp_polish_fetch_unsupported(ctx, u.off.data(), u.runs.data(), needed, &needed);
  }
  check_gp(ctx, rc, "gp_polish_fetch_unsupported");
  return u;
}

// name<TAB>start<TAB>end<TAB>k<K><TAB>kmers for the runs of record r (0 draft, 1 polished) of every input record whose
// emit[c] is set, by input record, then k in chain order, then start
inline void write_unsupported_bed(const std::string& path, const std::vector<std::string>& names, const std::vector<uint32_t>& ks,
                                  const UnsupportedRuns& u, uint32_t r, const std::vector<uint8_t>& emit)
{
  const size_t nk = ks.size();
  std::ofstream o(path);
  if (!o.good()) die("cannot write " + path);
  for (size_t c = 0; c < names.size(); c++) {
    if (!emit[c]) continue;
    for (size_t j = 0; j < nk; j++) {
      const size_t i = (c * 2 + r) * nk + j;
      for (uint64_t x = u.off[i]; x < u.off[i + 1]; x++)
        o << names[c] << '\t' << u.runs[x].start << '\t' << u.runs[x].end << "\tk" << ks[j] << '\t' << u.runs[x].kmers << '\n';
    }
  }
  if (!o.good()) die("cannot write " + path);
}

// ---------------------------------------------------------------------------------------
// FASTA/FASTQ reader with kseq semantics: gz or plain, multi-line sequences, name = text up
// to the first whitespace, comment = rest of the header line
// ---------------------------------------------------------------------------------------
struct FastaRecord {
  std::string name, comment, seq;
};

inline std::vector<FastaRecord> read_fasta(const std::string& path)
{
  gzFile f = gzopen(path.c_str(), "r");
  if (!f) die("cannot open " + path);
  std::string data;
  char buf[1 << 16];
  int n;
  while ((n = gzread(f, buf, sizeof buf)) > 0) data.append(buf, size_t(n));
  gzclose(f);
  std::vector<FastaRecord> recs;
  size_t i = 0;
  const size_t N = data.size();
  while (i < N) {
    while (i < N && data[i] != '>' && data[i] != '@') i++; // kseq skips to the next header mark
    if (i >= N) break;
    const bool fq = data[i] == '@';
    size_t e = data.find('\n', i);
    if (e == std::string::npos) e = N;
    std::string hdr = data.substr(i + 1, e - i - 1);
    if (!hdr.empty() && hdr.back() == '\r') hdr.pop_back();
    FastaRecord r;
    const size_t sp = hdr.find_first_of(" \t");
    r.name = hdr.substr(0, sp);
    if (sp != std::string::npos) {
      size_t c0 = sp + 1;
      r.comment = hdr.substr(c0);
    }
    i = e + 1;
    while (i < N && data[i] != '>' && data[i] != '+' && data[i] != '@') {
      size_t le = data.find('\n', i);
      if (le == std::string::npos) le = N;
      for (size_t q = i; q < le; q++) {
        const unsigned char c = (unsigned char)data[q];
        if (c > 32) r.seq.push_back((char)c); // kseq keeps printable, non-space characters
      }
      i = le + 1;
    }
    if (fq && i < N && data[i] == '+') { // skip the quality block (same length as the sequence)
      size_t le = data.find('\n', i);
      i = le == std::string::npos ? N : le + 1;
      size_t got = 0;
      while (i < N && got < r.seq.size()) {
        size_t le2 = data.find('\n', i);
        if (le2 == std::string::npos) le2 = N;
        got += le2 - i;
        i = le2 + 1;
      }
    }
    recs.push_back(std::move(r));
  }
  return recs;
}

} // namespace gph
