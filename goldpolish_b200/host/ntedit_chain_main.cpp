// goldpolish-ntedit (B200): drop-in for bcgsc/goldpolish scripts/goldpolish-ntedit.
// Same seven positionals (:3-16); the k chain (:20-29) runs inside ONE gp_polish call instead
// of one ntedit-gr process per k, then the 0.75 size guard (:31-40) picks the result.
// Only the final chain file is written (named as the script names it); the per-k
// intermediates of the script are not consumed by anything downstream.  GP_EDITS_VCF=1 also writes
// <outfile>.edits.vcf: what the whole chain changed, in draft coordinates (header only when the guard keeps the input).
// GP_KMER_QV=1 writes <outfile>.kmer_qv.tsv: k-mer completeness and QV of every record, draft and polished, for every k
// of the chain (when the guard keeps the input, the polished columns describe it).  GP_KMER_BED=1 writes
// <outfile>.kmer_unsupported.bed: the runs of unsupported k-mers of what <outfile> holds, for every k of the chain (the
// polished records, or the draft's runs when the guard keeps the input).
#include "gp_host.hpp"

#include <sys/stat.h>

using namespace gph;

static std::vector<std::string> split_ws(const std::string& s)
{
  std::istringstream in(s);
  std::vector<std::string> v;
  std::string t;
  while (in >> t) v.push_back(t);
  return v;
}

int main(int argc, char** argv)
{
  if (argc != 8) {
    std::cout << "Usage: goldpolish-ntedit <sequence fasta prefix> <ntHits BF filenames> <k values> <X parameter> "
                 "<Y parameter> <num threads> <output file>\n";
    return 1;
  }
  const std::string base = argv[1];
  const auto bfs = split_ws(argv[2]);
  const auto kstr = split_ws(argv[3]);
  const std::string X = argv[4], Y = argv[5], outfile = argv[7];
  if (bfs.size() != kstr.size() || bfs.empty() || bfs.size() > GP_MAX_K_VALUES) die("need one Bloom filter per k value");
  gp_config cfg;
  gp_default_config(&cfg); // -d5 -i5 -m1 -a1 (:27)
  cfg.nk = uint32_t(bfs.size());
  cfg.missing_ratio = std::stof(X);
  cfg.edit_ratio = std::stof(Y);
  cfg.use_ratio = 1;
  std::vector<uint8_t> all_payload, one;
  for (size_t i = 0; i < bfs.size(); i++) {
    const auto h = bf_format::load(bfs[i], one);
    if (h.hash_num != GP_HASH_NUM || h.bytes != GP_BF_BYTES) die("unsupported Bloom filter geometry in " + bfs[i]);
    cfg.k[i] = h.k; // ntedit-gr takes k from the filter header, not from the K list (ntedit.cpp:2022)
    all_payload.insert(all_payload.end(), one.begin(), one.end());
  }
  if (const char* d = std::getenv("GP_DEVICE")) cfg.device = std::atoi(d);
  const char* vcf_env = std::getenv("GP_EDITS_VCF");
  cfg.track_edits = vcf_env && std::string(vcf_env) == "1";
  const char* qv_env = std::getenv("GP_KMER_QV");
  const char* bed_env = std::getenv("GP_KMER_BED");
  const bool kmer_qv = qv_env && std::string(qv_env) == "1", kmer_bed = bed_env && std::string(bed_env) == "1";
  cfg.kmer_support = kmer_qv || kmer_bed;
  const std::string in_path = base + ".fa";
  struct stat st;
  if (stat(in_path.c_str(), &st) != 0) die("cannot stat " + in_path);
  const uint64_t input_size = uint64_t(st.st_size);
  const auto recs = read_fasta(in_path);
  std::string all;
  std::vector<uint64_t> off(1, 0);
  for (const auto& r : recs) { all += r.seq; off.push_back(all.size()); }
  std::vector<uint32_t> cb(recs.size(), 0);
  gp_ctx* ctx = nullptr;
  if (gp_ctx_create(&cfg, &ctx) != GP_OK) die(std::string("gp_ctx_create: ") + gp_last_error(nullptr));
  check_gp(ctx, gp_filters_load(ctx, 1, all_payload.data()), "gp_filters_load");
  std::vector<char> out(all.size() + all.size() / 2 + 65536);
  std::vector<uint64_t> ooff(recs.size() + 1);
  std::vector<uint8_t> dropped(recs.size() + 1);
  int rc = gp_polish(ctx, uint32_t(recs.size()), all.data(), off.data(), cb.data(), out.data(), out.size(), ooff.data(), dropped.data());
  if (rc == GP_ERR_ARG && ooff[recs.size()] > out.size()) {
    out.resize(ooff[recs.size()]);
    rc = gp_polish_fetch(ctx, out.data(), out.size(), ooff.data(), dropped.data());
  }
  check_gp(ctx, rc, "gp_polish");
  EditRecords er;
  if (cfg.track_edits) er = fetch_edits(ctx, uint32_t(recs.size()));
  KmerSupport ks;
  if (kmer_qv) ks = fetch_support(ctx, uint32_t(recs.size()), cfg.nk, 1);
  UnsupportedRuns ur;
  if (kmer_bed) ur = fetch_unsupported(ctx, uint32_t(recs.size()), cfg.nk);
  gp_ctx_destroy(ctx);
  // the chain's last file, named as the script's loop names it (:27-28)
  std::string prev = base;
  for (const auto& k : kstr) prev += ".k" + k + ".X" + X + ".Y" + Y + "_edited";
  uint64_t output_size = 0;
  {
    std::ofstream o(prev + ".fa");
    for (size_t i = 0; i < recs.size(); i++) {
      if (dropped[i]) continue;
      std::string hdr = ">" + recs[i].name + (recs[i].comment.empty() ? "" : " " + recs[i].comment) + "\n";
      o << hdr;
      o.write(out.data() + ooff[i], std::streamsize(ooff[i + 1] - ooff[i]));
      o << "\n";
      output_size += hdr.size() + (ooff[i + 1] - ooff[i]) + 1;
    }
  }
  std::remove(outfile.c_str());
  if (const char* bed = std::getenv("GP_FLAGGED_BED")) { // the flagged regions of what <outfile> will hold
    const bool rejected = gp_guard_rejects(input_size, output_size) != 0;
    std::vector<std::string> names;
    std::vector<uint64_t> eoff(1, 0);
    std::string eseq;
    for (size_t i = 0; i < recs.size(); i++) {
      if (!rejected && dropped[i]) continue;
      names.push_back(recs[i].name);
      if (rejected) eseq += recs[i].seq;
      else eseq.append(out.data() + ooff[i], size_t(ooff[i + 1] - ooff[i]));
      eoff.push_back(eseq.size());
    }
    write_flagged_bed(bed, names, eseq.data(), eoff);
  }
  if (cfg.track_edits) { // the edits of the whole k chain, of what <outfile> will hold: none when the guard keeps the input
    std::vector<std::string> names;
    std::vector<uint64_t> lens;
    for (size_t i = 0; i < recs.size(); i++) { names.push_back(recs[i].name); lens.push_back(off[i + 1] - off[i]); }
    write_edits_vcf(outfile + ".edits.vcf", names, lens, gp_guard_rejects(input_size, output_size) ? nullptr : &er);
  }
  if (kmer_bed) { // the runs of what <outfile> will hold: the polished records, or the input when the guard keeps it
    const bool rejected = gp_guard_rejects(input_size, output_size) != 0;
    std::vector<std::string> names;
    std::vector<uint8_t> emit;
    for (size_t i = 0; i < recs.size(); i++) { names.push_back(recs[i].name); emit.push_back(rejected || !dropped[i] ? 1 : 0); }
    write_unsupported_bed(outfile + ".kmer_unsupported.bed", names, std::vector<uint32_t>(cfg.k, cfg.k + cfg.nk), ur,
                          rejected ? 0 : 1, emit);
  }
  if (kmer_qv) {
    std::vector<std::string> names;
    for (const auto& r : recs) names.push_back(r.name);
    write_kmer_qv(outfile + ".kmer_qv.tsv", names, std::vector<uint32_t>(cfg.k, cfg.k + cfg.nk), ks,
                  gp_guard_rejects(input_size, output_size) != 0);
  }
  if (gp_guard_rejects(input_size, output_size)) { // :31-37
    if (symlink(in_path.c_str(), outfile.c_str()) != 0) die("symlink failed");
    std::cout << "goldpolish-ntedit: skipped " << in_path << "\n";
  } else if (symlink((prev + ".fa").c_str(), outfile.c_str()) != 0) die("symlink failed");
  return 0;
}
