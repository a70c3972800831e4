// goldpolish-targeted-bfs (B200): drop-in for bcgsc/goldpolish src/goldpolish_targeted_bfs.cpp.
//
// Same argv (:250-268), same named-pipe protocol in the current directory (:148-244), same
// "<batch>-k<K>.bf" outputs (:79-84,138-140).  Differences are internal only:
//   * the mapped reads are put on the GPU(s) once, 2-bit packed, streamed from the reads file in slabs (the host
//     never holds the read set as text; the reference re-reads a read from the file for every use, seqindex.hpp:59-102);
//   * batch requests that are pending at the same time are built by ONE gp_build_filters call per GPU;
//   * batches are served by a bounded pool of workers (the reference: OpenMP tasks on `threads` threads, :177-192,
//     223-224), never one thread per batch;
//   * a client may append "@polish <batch.fa> <out.fa>" to its target ids (goldpolish_b200's goldpolish-polish-batch
//     does): the batch is then polished in the same GPU pass that builds its filters, and <out.fa> is what
//     goldpolish-ntedit would have produced from the .bf files (k chain + 0.75 guard);
//   * GP_DEVICES=0,1,... (or GP_DEVICE=n) names the GPUs: one context and one GPU thread per device, every request goes
//     to the device with the fewest read bases pending.  Batches are independent (:70-77), so nothing is exchanged
//     between devices and the answers travel back through the same FIFOs.
#include "gp_host.hpp"

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>

#include <sys/stat.h>
#include <sys/types.h>

using namespace gph;

namespace {

const unsigned MX_THRESHOLD_MIN = 1, MX_THRESHOLD_MAX = 30; // :34-35
const std::string BATCH_NAME_INPUT_PIPE = "batch_name_input";
const std::string BATCH_TARGET_IDS_INPUT_READY_PIPE = "batch_target_ids_input_ready";
const std::string END_SYMBOL = "x";

void make_pipe(const std::string& p)
{ // src/utils.cpp:72-78
  if (mkfifo(p.c_str(), S_IRUSR | S_IWUSR) != 0) die("mkfifo failed: " + std::string(std::strerror(errno)));
}
std::string read_pipe(const std::string& p)
{ // :80-87
  std::string s;
  std::ifstream in(p);
  in >> s;
  return s;
}
void confirm_pipe(const std::string& p)
{ // :89-94
  std::ofstream o(p);
  o << "1" << std::endl;
}
void bind_to_parent()
{ // :55-70
  std::thread([] {
    while (getppid() != 1) std::this_thread::sleep_for(std::chrono::seconds(1));
    std::exit(EXIT_FAILURE);
  }).detach();
}

struct Request {
  std::string batch;
  std::vector<gp_read_entry> entries;
  uint64_t bases = 0;            // read bases to hash (the load estimate)
  std::vector<uint8_t> payload;  // nk * GP_BF_BYTES once built
  bool done = false;
  // "@polish <batch.fa> <out.fa>" after the target ids (goldpolish_b200's own goldpolish-polish-batch sends it): the
  // batch's contigs are polished in the same GPU pass as its filters are built (gp_pipeline_run) -- what
  // goldpolish-make's `%.ntedited.fa` rule would do with goldpolish-ntedit and four ntedit-gr processes
  bool polish = false;
  std::string seqs_path, out_path;
  std::vector<FastaRecord> recs;
  std::vector<std::string> polished;   // one per record ("" + dropped flag when the reference would not emit it)
  std::vector<uint8_t> dropped;
  uint64_t input_size = 0;             // bytes of <batch.fa> (the guard compares file sizes, scripts/goldpolish-ntedit:31-37)
  std::string body;                    // what goes to <out.fa> ...
  bool keep_input = false;             // ... unless the guard rejected it: then <out.fa> is a copy of <batch.fa>
  // "@prep <k> <prepd.fa>" after "@polish": also leave what `goldpolish-mask -s -k<k> <out.fa>` would print
  // (scripts/goldpolish-make:65-66) in <prepd.fa>, masked on the device (gp_prep) while the records are at hand
  unsigned prep_k = 0;
  std::string prep_path, prep_body;
};

// ">id[ comment]\n" + sequence + "\n", as ntEdit (ntedit.cpp:1853-1856) and btllib::SeqWriter write FASTA
void append_record(std::string& body, const FastaRecord& rec, const char* seq, size_t len)
{
  body += ">" + rec.name + (rec.comment.empty() ? "" : " " + rec.comment) + "\n";
  body.append(seq, len);
  body += "\n";
}

// One GPU: a context, the read store, a queue of pending requests and the thread that builds them.
struct Device {
  int ordinal = 0;
  gp_ctx* ctx = nullptr;
  std::vector<unsigned> ks;
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  std::deque<std::shared_ptr<Request>> queue;
  uint64_t pending_bases = 0;
  uint64_t batches_served = 0;
  bool stopping = false;
  std::thread thread;

  // <out.fa> of every polished request (k chain + the 0.75 guard), and <prepd.fa> of those that asked for it: the
  // records that <out.fa> holds, masked by ONE gp_prep call for all of them
  void finish_polished(std::vector<std::shared_ptr<Request>>& todo)
  {
    std::string mseqs;
    std::vector<uint64_t> moff(1, 0);
    struct Ref { Request* r; const FastaRecord* rec; };
    std::vector<Ref> mrecs;
    std::vector<FastaRecord> reread; // (records of guard-rejected batches are masked as the input file holds them)
    for (auto& rp : todo) {
      Request& r = *rp;
      if (!r.polish) continue;
      for (size_t i = 0; i < r.recs.size(); i++)
        if (!r.dropped[i]) append_record(r.body, r.recs[i], r.polished[i].data(), r.polished[i].size()); // ntedit.cpp:1850
      const bool keep_input = r.keep_input = gp_guard_rejects(r.input_size, r.body.size()) != 0; // scripts/goldpolish-ntedit:31-37
      if (r.prep_k == 0) continue;
      for (size_t i = 0; i < r.recs.size(); i++) {
        if (!keep_input && r.dropped[i]) continue;
        const std::string& seq = keep_input ? r.recs[i].seq : r.polished[i];
        mseqs += seq;
        moff.push_back(mseqs.size());
        mrecs.push_back(Ref{ &r, &r.recs[i] });
      }
    }
    if (mrecs.empty()) return;
    // all requests of a call share one mask width in practice (the first k value); group by k to be exact
    std::vector<unsigned> widths;
    for (const auto& m : mrecs)
      if (std::find(widths.begin(), widths.end(), m.r->prep_k) == widths.end()) widths.push_back(m.r->prep_k);
    for (const unsigned kk : widths) {
      std::string seqs;
      std::vector<uint64_t> off(1, 0);
      std::vector<size_t> who;
      for (size_t i = 0; i < mrecs.size(); i++)
        if (mrecs[i].r->prep_k == kk) {
          seqs.append(mseqs, moff[i], moff[i + 1] - moff[i]);
          off.push_back(seqs.size());
          who.push_back(i);
        }
      std::vector<char> out(seqs.size() + who.size() + 16);
      std::vector<uint64_t> ooff(who.size() + 1, 0);
      check_gp(ctx, gp_prep(ctx, uint32_t(who.size()), seqs.data(), off.data(), 1, kk, 0, out.data(), out.size(), ooff.data()),
               "gp_prep");
      for (size_t j = 0; j < who.size(); j++)
        append_record(mrecs[who[j]].r->prep_body, *mrecs[who[j]].rec, out.data() + ooff[j], size_t(ooff[j + 1] - ooff[j]));
    }
  }

  // builds every request that is pending in one call.  The payloads land in page-locked memory that the build
  // kernel fills filter by filter as they become final (gp_build_output_host): no bulk copy after the build, and
  // what bfs[i]->save() writes (:138-140) is ready when the call returns.
  void loop()
  {
    uint8_t* pinned = nullptr;
    size_t pinned_cap = 0;
    const size_t max_per_call = 4096; // (bounds the page-locked buffer: 8 GiB)
    for (;;) {
      std::vector<std::shared_ptr<Request>> todo;
      {
        std::unique_lock<std::mutex> lk(mu);
        cv_work.wait(lk, [&] { return stopping || !queue.empty(); });
        if (queue.empty() && stopping) { gp_build_output_host(ctx, nullptr); gp_host_free(pinned); return; }
        while (!queue.empty() && todo.size() < max_per_call) { todo.push_back(queue.front()); queue.pop_front(); }
      }
      std::vector<uint64_t> off(1, 0);
      std::vector<gp_read_entry> ents;
      for (const auto& r : todo) {
        ents.insert(ents.end(), r->entries.begin(), r->entries.end());
        off.push_back(ents.size());
      }
      const size_t need = todo.size() * ks.size() * GP_BF_BYTES;
      std::vector<uint8_t> pageable;
      uint8_t* out = nullptr;
      if (need > pinned_cap) {
        gp_build_output_host(ctx, nullptr);
        gp_host_free(pinned);
        pinned_cap = need + need / 2;
        pinned = static_cast<uint8_t*>(gp_host_alloc(pinned_cap));
        if (!pinned) pinned_cap = 0;
        else check_gp(ctx, gp_build_output_host(ctx, pinned), "gp_build_output_host");
      }
      if (pinned) out = pinned;
      else { pageable.resize(need); out = pageable.data(); } // no page-locked memory to be had: plain copy
      bool any_polish = false;
      for (const auto& r : todo) any_polish |= r->polish;
      if (!any_polish) {
        check_gp(ctx, gp_build_filters(ctx, uint32_t(todo.size()), off.data(), ents.data(), out), "gp_build_filters");
      } else {
        // filters of every request + the k chain over the contigs of those that asked for it, as one overlapped pass
        std::string seqs;
        std::vector<uint64_t> coff(1, 0);
        std::vector<uint32_t> cbatch;
        for (size_t i = 0; i < todo.size(); i++)
          if (todo[i]->polish)
            for (const auto& rec : todo[i]->recs) { seqs += rec.seq; coff.push_back(seqs.size()); cbatch.push_back(uint32_t(i)); }
        check_gp(ctx, gp_build_stage(ctx, uint32_t(todo.size()), off.data(), ents.data()), "gp_build_stage");
        check_gp(ctx, gp_polish_stage(ctx, uint32_t(cbatch.size()), seqs.data(), coff.data(), cbatch.data()), "gp_polish_stage");
        check_gp(ctx, gp_pipeline_run(ctx), "gp_pipeline_run");
        check_gp(ctx, gp_build_fetch(ctx, out), "gp_build_fetch");
        std::vector<char> pout(seqs.size() + seqs.size() / 2 + 65536);
        std::vector<uint64_t> poff(cbatch.size() + 1);
        std::vector<uint8_t> dropped(cbatch.size() + 1);
        int rc = gp_polish_fetch(ctx, pout.data(), pout.size(), poff.data(), dropped.data());
        if (rc == GP_ERR_ARG && poff[cbatch.size()] > pout.size()) {
          pout.resize(poff[cbatch.size()]);
          rc = gp_polish_fetch(ctx, pout.data(), pout.size(), poff.data(), dropped.data());
        }
        check_gp(ctx, rc, "gp_polish_fetch");
        size_t c = 0;
        for (size_t i = 0; i < todo.size(); i++)
          if (todo[i]->polish)
            for (size_t j = 0; j < todo[i]->recs.size(); j++, c++) {
              todo[i]->polished.emplace_back(pout.data() + poff[c], size_t(poff[c + 1] - poff[c]));
              todo[i]->dropped.push_back(dropped[c]);
            }
        finish_polished(todo);
      }
      {
        std::lock_guard<std::mutex> lk(mu);
        for (size_t i = 0; i < todo.size(); i++) {
          todo[i]->payload.assign(out + i * ks.size() * GP_BF_BYTES, out + (i + 1) * ks.size() * GP_BF_BYTES);
          todo[i]->done = true;
          pending_bases -= todo[i]->bases;
        }
        batches_served += todo.size();
      }
      cv_done.notify_all();
    }
  }
};

// A fixed number of workers serve the batches (serve_batch, :55-146): read the target ids from the batch's pipe, select
// the reads, hand the request to a device, write the .bf files, acknowledge.
struct Pool {
  std::mutex mu;
  std::condition_variable cv;
  std::deque<std::string> batches;
  bool closing = false;
  std::vector<std::thread> workers;
};

std::vector<int> device_list()
{
  std::vector<int> v;
  if (const char* e = std::getenv("GP_DEVICES")) {
    std::stringstream ss(e);
    std::string tok;
    while (std::getline(ss, tok, ',')) {
      if (tok.empty()) continue;
      char* end = nullptr;
      const long d = std::strtol(tok.c_str(), &end, 10);
      if (*end != '\0' || d < 0) die("GP_DEVICES must be a comma-separated list of CUDA ordinals, got '" + std::string(e) + "'");
      v.push_back(int(d));
    }
  }
  if (v.empty()) v.push_back(std::getenv("GP_DEVICE") ? std::atoi(std::getenv("GP_DEVICE")) : 0);
  return v;
}

} // namespace

int main(int argc, char** argv)
{
  if (argc < 8) die("Wrong args."); // :253
  bind_to_parent();
  int a = 1;
  const std::string target_seqs = argv[a++], target_index_path = argv[a++], mappings_path = argv[a++];
  const std::string reads_path = argv[a++], reads_index_path = argv[a++];
  const double mx_max_per_10kbp = std::stod(argv[a++]);
  const double subsample_max_per_10kbp = std::stod(argv[a++]);
  const int threads = std::stoi(argv[a++]);
  std::vector<unsigned> ks;
  while (a < argc) ks.push_back(unsigned(std::stoi(argv[a++])));
  if (ks.empty() || ks.size() > GP_MAX_K_VALUES) die("need 1..8 k values");
  for (const unsigned k : ks) // the device keeps a k-mer in one 64-bit word of packed bases
    if (k < 4 || k > 32) die("k = " + std::to_string(k) + " is not supported: k must be within 4..32");

  info("Loading index from " + target_index_path);
  const SeqIndex targets = SeqIndex::load(target_index_path, target_seqs);
  info("Loading index from " + reads_index_path);
  const SeqIndex reads = SeqIndex::load(reads_index_path, reads_path);
  info("Loading mappings from " + mappings_path);
  const Mappings maps(mappings_path, targets, MX_THRESHOLD_MIN, MX_THRESHOLD_MAX, mx_max_per_10kbp);

  gp_config cfg;
  gp_default_config(&cfg);
  cfg.nk = uint32_t(ks.size());
  for (size_t i = 0; i < ks.size(); i++) cfg.k[i] = ks[i];
  std::vector<std::unique_ptr<Device>> devs;
  for (const int ord : device_list()) {
    auto d = std::make_unique<Device>();
    d->ordinal = ord;
    d->ks = ks;
    cfg.device = ord;
    if (gp_ctx_create(&cfg, &d->ctx) != GP_OK) die("gp_ctx_create (device " + std::to_string(ord) + "): " + gp_last_error(nullptr));
    devs.push_back(std::move(d));
  }

  // every read that some target maps goes to every device once (SeqIndex::get_seq<1> re-reads per use), streamed from
  // the file in slabs: the host holds one slab of text at a time
  std::unordered_map<std::string, uint32_t> read_slot;
  {
    std::vector<const std::string*> order;
    std::vector<uint32_t> lens;
    uint64_t total = 0;
    maps.for_each([&](const std::string&, const std::vector<std::string>& ids) {
      for (const auto& id : ids)
        if (read_slot.emplace(id, uint32_t(order.size())).second) {
          order.push_back(&id);
          lens.push_back(uint32_t(reads.at(id).len));
          total += lens.back();
        }
    });
    info("Uploading " + std::to_string(order.size()) + " mapped reads (" + std::to_string(total) + " bases) to " +
         std::to_string(devs.size()) + " device(s)");
    for (auto& d : devs) check_gp(d->ctx, gp_reads_begin(d->ctx, order.size(), lens.data()), "gp_reads_begin");
    // slabs of ~64 MiB of consecutive reads, each read from the file by all host cores (SeqIndex::read_many)
    const uint64_t slab_bytes = 64u << 20;
    std::string slab;
    for (size_t first = 0; first < order.size();) {
      size_t n = 0;
      uint64_t bytes = 0;
      while (first + n < order.size() && (n == 0 || bytes + lens[first + n] <= slab_bytes)) bytes += lens[first + n++];
      reads.read_many(order, first, n, slab);
      for (auto& d : devs) check_gp(d->ctx, gp_reads_append(d->ctx, slab.data(), n), "gp_reads_append");
      first += n;
    }
    for (auto& d : devs) check_gp(d->ctx, gp_reads_end(d->ctx), "gp_reads_end");
  }

  make_pipe(BATCH_NAME_INPUT_PIPE);
  make_pipe(BATCH_TARGET_IDS_INPUT_READY_PIPE);
  info("Accepting batch names at " + BATCH_NAME_INPUT_PIPE);
  for (auto& d : devs) d->thread = std::thread(&Device::loop, d.get());

  auto serve_batch = [&](const std::string& batch) { // :55-146
    const std::string ids_pipe = batch + "-target_ids_input", ready_pipe = batch + "-bfs_ready";
    auto req = std::make_shared<Request>();
    req->batch = batch;
    {
      std::ifstream in(ids_pipe);
      std::string id;
      while (bool(in >> id) && id != END_SYMBOL) {
        if (id == "@polish") { // (not a valid FASTA id: '@' opens a FASTQ header)
          if (!(in >> req->seqs_path >> req->out_path)) die("malformed @polish request for batch " + batch);
          req->polish = true;
          continue;
        }
        if (id == "@prep") {
          long kk = 0;
          if (!(in >> kk >> req->prep_path) || kk < 1 || kk > 64) die("malformed @prep request for batch " + batch);
          req->prep_k = unsigned(kk);
          continue;
        }
        const uint64_t tlen = targets.at(id).len;
        const auto& mapped = maps.get(id);
        if (mapped.empty()) continue;
        const Selection sel = select_reads(mapped, reads, tlen, subsample_max_per_10kbp);
        for (const auto& r : sel.reads) {
          req->entries.push_back(gp_read_entry{ read_slot.at(r), uint32_t(sel.kmer_threshold) });
          req->bases += reads.at(r).len;
        }
      }
    }
    if (req->prep_k && !req->polish) die("@prep without @polish for batch " + batch);
    if (req->polish) {
      struct stat st;
      if (stat(req->seqs_path.c_str(), &st) != 0) die("cannot stat " + req->seqs_path);
      req->input_size = uint64_t(st.st_size);
      req->recs = read_fasta(req->seqs_path);
    }
    // the device with the least work pending
    Device* dev = devs[0].get();
    if (devs.size() > 1) {
      uint64_t best = ~0ull;
      for (auto& d : devs) {
        std::lock_guard<std::mutex> lk(d->mu);
        if (d->pending_bases < best) { best = d->pending_bases; dev = d.get(); }
      }
    }
    {
      std::unique_lock<std::mutex> lk(dev->mu);
      dev->pending_bases += req->bases;
      dev->queue.push_back(req);
      dev->cv_work.notify_one();
      dev->cv_done.wait(lk, [&] { return req->done; });
    }
    for (size_t i = 0; i < ks.size(); i++)
      bf_format::save(batch + "-k" + std::to_string(ks[i]) + ".bf", req->payload.data() + i * GP_BF_BYTES, GP_BF_BYTES,
                      GP_HASH_NUM, ks[i]);
    if (req->polish) { // after the .bf files: `make` must not find the polished file older than its prerequisites
      {
        std::ofstream o(req->out_path, std::ios::binary);
        if (!o.good()) die("cannot write " + req->out_path);
        if (req->keep_input) { // scripts/goldpolish-ntedit:31-37
          std::ifstream in(req->seqs_path, std::ios::binary);
          o << in.rdbuf();
        } else o << req->body;
      }
      if (req->prep_k) { // after <out.fa>, its prerequisite in goldpolish-make's `%.prepd.fa: %.fa`
        std::ofstream o(req->prep_path, std::ios::binary);
        if (!o.good()) die("cannot write " + req->prep_path);
        o << req->prep_body;
      }
    }
    confirm_pipe(ready_pipe);
    std::remove(ids_pipe.c_str());
    std::remove(ready_pipe.c_str());
  };

  // The workers mostly wait -- for a client to write its ids, for the GPU -- so there are more of them than the
  // `threads` the reference computes with; the number of batches in flight, and with it the size of a GPU call, is
  // bounded by it.  GP_SERVER_WORKERS overrides.
  size_t n_workers = size_t(std::max(2, threads)) * 4;
  if (n_workers > 256) n_workers = 256;
  if (const char* e = std::getenv("GP_SERVER_WORKERS")) n_workers = size_t(std::max(1, std::atoi(e)));
  Pool pool;
  for (size_t w = 0; w < n_workers; w++)
    pool.workers.emplace_back([&] {
      for (;;) {
        std::string batch;
        {
          std::unique_lock<std::mutex> lk(pool.mu);
          pool.cv.wait(lk, [&] { return pool.closing || !pool.batches.empty(); });
          if (pool.batches.empty()) return;
          batch = std::move(pool.batches.front());
          pool.batches.pop_front();
        }
        serve_batch(batch);
      }
    });
  for (;;) { // process_batch_name, :148-195
    const std::string batch = read_pipe(BATCH_NAME_INPUT_PIPE);
    if (batch.empty() || batch == END_SYMBOL) break;
    make_pipe(batch + "-target_ids_input");
    make_pipe(batch + "-bfs_ready");
    confirm_pipe(BATCH_TARGET_IDS_INPUT_READY_PIPE);
    {
      std::lock_guard<std::mutex> lk(pool.mu);
      pool.batches.push_back(batch);
    }
    pool.cv.notify_one();
  }
  {
    std::lock_guard<std::mutex> lk(pool.mu);
    pool.closing = true;
  }
  pool.cv.notify_all();
  for (auto& w : pool.workers) w.join();
  for (auto& d : devs) {
    {
      std::lock_guard<std::mutex> lk(d->mu);
      d->stopping = true;
    }
    d->cv_work.notify_all();
    d->thread.join();
    info("device " + std::to_string(d->ordinal) + ": " + std::to_string(d->batches_served) + " batches served");
    gp_ctx_destroy(d->ctx);
  }
  std::remove(BATCH_NAME_INPUT_PIPE.c_str());
  std::remove(BATCH_TARGET_IDS_INPUT_READY_PIPE.c_str());
  info("Targeted BF builder done!");
  return 0;
}
