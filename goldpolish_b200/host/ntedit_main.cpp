// ntedit-gr (B200): drop-in for the ntEdit fork of bcgsc/goldpolish (subprojects/ntedit/
// ntedit.cpp main :1869-2124, readAndCorrect :1774-1867).  Same options; the scan / edit loop
// runs on the GPU through gp_polish.  Unsupported on purpose (exit 1 with a message): -s 1 (SNV
// mode) and -e (secondary filter), both marked EXPERIMENTAL upstream and unused by GoldPolish.
#include "gp_host.hpp"

#include <getopt.h>

using namespace gph;

namespace {
const char* PROGRAM = "ntedit";
const char shortopts[] = "t:f:s:k:z:b:r:v:d:i:X:Y:x:y:m:c:j:s:e:a:"; // ntedit.cpp:116
const struct option longopts[] = {                                   // :124-147
  { "threads", required_argument, nullptr, 't' }, { "draft_file", required_argument, nullptr, 'f' },
  { "k", required_argument, nullptr, 'k' }, { "minimum_contig_length", required_argument, nullptr, 'z' },
  { "maximum_insertions", required_argument, nullptr, 'i' }, { "maximum_deletions", required_argument, nullptr, 'd' },
  { "insertion_cap", required_argument, nullptr, 'c' }, { "edit_threshold", required_argument, nullptr, 'y' },
  { "missing_threshold", required_argument, nullptr, 'x' }, { "edit_ratio", required_argument, nullptr, 'Y' },
  { "missing_ratio", required_argument, nullptr, 'X' }, { "jump", required_argument, nullptr, 'j' },
  { "bloom_filename", required_argument, nullptr, 'r' }, { "bloomrep_filename", required_argument, nullptr, 'e' },
  { "outfile_prefix", required_argument, nullptr, 'b' }, { "mode", required_argument, nullptr, 'm' },
  { "snv", required_argument, nullptr, 's' }, { "mask", required_argument, nullptr, 'a' },
  { "verbose", required_argument, nullptr, 'v' }, { "help", no_argument, nullptr, 1 },
  { "version", no_argument, nullptr, 2 },
  { "bed", required_argument, nullptr, 3 }, // extension: write the flagged (soft-masked, -a1) regions as BED rows
  { "vcf", required_argument, nullptr, 4 }, // extension: write what polishing changed as VCF records (draft coordinates)
  { nullptr, 0, nullptr, 0 }
};
void assert_readable(const std::string& p)
{ // :346-353
  if (access(p.c_str(), R_OK) == -1) {
    std::cerr << PROGRAM << ": error: `" << p << "': " << std::strerror(errno) << std::endl;
    std::exit(EXIT_FAILURE);
  }
}
} // namespace

int main(int argc, char** argv)
{
  gp_config cfg;
  gp_default_config(&cfg);
  cfg.max_insertions = 5; cfg.max_deletions = 5; cfg.mode = 0; cfg.mask = 0; // ntedit.cpp:86-87,109,111
  cfg.use_ratio = 0;
  std::string draft, bloom, bloomrep, prefix, bed, vcf;
  unsigned nthreads = 1;
  int snv = 0, verbose = 0;
  bool dieflag = false;
  for (int c; (c = getopt_long(argc, argv, shortopts, longopts, nullptr)) != -1;) {
    std::istringstream arg(optarg != nullptr ? optarg : "");
    float cap_ignored;
    switch (c) {
    case '?': dieflag = true; break;
    case 't': arg >> nthreads; break;
    case 'f': arg >> draft; break;
    case 'z': arg >> cfg.min_contig_len; break;
    case 'b': arg >> prefix; break;
    case 'r': arg >> bloom; break;
    case 'e': arg >> bloomrep; break;
    case 'd': arg >> cfg.max_deletions; break;
    case 'i': arg >> cfg.max_insertions; break;
    case 'x': arg >> cfg.missing_threshold; break;
    case 'y': arg >> cfg.edit_threshold; break;
    case 'X': arg >> cfg.missing_ratio; cfg.use_ratio = 1; break; // :1909-1912
    case 'Y': arg >> cfg.edit_ratio; cfg.use_ratio = 1; break;
    case 'c': arg >> cap_ignored; break; // overwritten with k*1.5 at :2024-2025
    case 'j': arg >> cfg.jump; break;
    case 'm': arg >> cfg.mode; break;
    case 's': arg >> snv; break;
    case 'a': arg >> cfg.mask; break;
    case 'v': arg >> verbose; break;
    case 1: std::cerr << "ntedit v1.3.5 (goldpolish_b200 GPU drop-in)\n"; return 0;
    case 2: std::cerr << "ntedit version 1.3.5 (goldpolish_b200 GPU drop-in)\n"; return 0;
    case 3: arg >> bed; break;
    case 4: arg >> vcf; break;
    default: break;
    }
    if (optarg != nullptr && (!arg.eof() || arg.fail())) { // :1944-1947
      std::cerr << PROGRAM << ": invalid option: `-" << char(c) << optarg << "'\n";
      return EXIT_FAILURE;
    }
  }
  if (draft.empty()) { std::cerr << PROGRAM << ": error: need to specify assembly draft file (-f)\n"; dieflag = true; }
  else assert_readable(draft);
  if (bloom.empty()) { std::cerr << PROGRAM << ": error: need to specify the bloom filter file (-r)\n"; dieflag = true; }
  else assert_readable(bloom);
  if (dieflag) { std::cerr << "Try `" << PROGRAM << " --help' for more information.\n"; return EXIT_FAILURE; }
  if (snv || !bloomrep.empty()) die("-s 1 and -e are EXPERIMENTAL upstream and not offered by the GPU drop-in");
  (void)nthreads; (void)verbose;

  std::vector<uint8_t> payload;
  const bf_format::Header h = bf_format::load(bloom, payload);
  if (h.hash_num == 0) { std::cerr << PROGRAM << ": error: Bloom filter file supplied (-r) is incorrect.\n"; return EXIT_FAILURE; }
  if (h.hash_num != GP_HASH_NUM || h.bytes != GP_BF_BYTES)
    die("the GPU drop-in handles GoldPolish's filter geometry only (4 hashes, 512 KiB); got " +
        std::to_string(h.hash_num) + " hashes, " + std::to_string(h.bytes) + " bytes");
  cfg.nk = 1;
  cfg.k[0] = h.k; // :2022
  // parameter fix-ups of :2045-2060
  if ((cfg.max_insertions == 0 && cfg.max_deletions > 0) || (cfg.max_insertions == 1 && cfg.max_deletions > 1)) {
    std::cerr << PROGRAM << ": warning: i and d parameter combination is not possible; d was set to the value of i.\n";
    cfg.max_deletions = cfg.max_insertions;
  }
  if (cfg.max_insertions > 5) cfg.max_insertions = 5;
  if (cfg.max_deletions > 10) cfg.max_deletions = 10;
  if (prefix.empty()) { // :2063-2069
    const std::string db = draft.substr(draft.find_last_of("/\\") + 1), bb = bloom.substr(bloom.find_last_of("/\\") + 1);
    std::ostringstream o;
    o << db << "_k" << h.k << "_z" << cfg.min_contig_len << "_r" << bb << "_i" << cfg.max_insertions << "_d"
      << cfg.max_deletions << "_m" << cfg.mode;
    prefix = o.str();
  }
  if (const char* d = std::getenv("GP_DEVICE")) cfg.device = std::atoi(d);
  cfg.track_edits = vcf.empty() ? 0 : 1;

  const std::vector<FastaRecord> recs = read_fasta(draft);
  std::string all;
  std::vector<uint64_t> off(1, 0);
  for (const auto& r : recs) { all += r.seq; off.push_back(all.size()); }
  std::vector<uint32_t> cb(recs.size(), 0);
  gp_ctx* ctx = nullptr;
  if (gp_ctx_create(&cfg, &ctx) != GP_OK) die(std::string("gp_ctx_create: ") + gp_last_error(nullptr));
  check_gp(ctx, gp_filters_load(ctx, 1, payload.data()), "gp_filters_load");
  std::vector<char> out(all.size() + all.size() / 2 + 65536);
  std::vector<uint64_t> ooff(recs.size() + 1);
  std::vector<uint8_t> dropped(recs.size() + 1);
  int rc = gp_polish(ctx, uint32_t(recs.size()), all.data(), off.data(), cb.data(), out.data(), out.size(), ooff.data(), dropped.data());
  if (rc == GP_ERR_ARG && ooff[recs.size()] > out.size()) {
    out.resize(ooff[recs.size()]);
    rc = gp_polish_fetch(ctx, out.data(), out.size(), ooff.data(), dropped.data());
  }
  check_gp(ctx, rc, "gp_polish");
  std::ofstream o(prefix + "_edited.fa"); // :1785
  for (size_t i = 0; i < recs.size(); i++) {
    if (dropped[i]) continue; // :1850
    o << ">" << recs[i].name;
    if (!recs[i].comment.empty()) o << " " << recs[i].comment; // :1832-1837
    o << "\n";
    o.write(out.data() + ooff[i], std::streamsize(ooff[i + 1] - ooff[i]));
    o << "\n";
  }
  if (bed.empty() && std::getenv("GP_FLAGGED_BED")) bed = std::getenv("GP_FLAGGED_BED");
  if (!bed.empty()) { // emitted records only, coordinates of the polished record
    std::vector<std::string> names;
    std::vector<uint64_t> eoff(1, 0);
    std::string eseq;
    for (size_t i = 0; i < recs.size(); i++) {
      if (dropped[i]) continue;
      names.push_back(recs[i].name);
      eseq.append(out.data() + ooff[i], size_t(ooff[i + 1] - ooff[i]));
      eoff.push_back(eseq.size());
    }
    write_flagged_bed(bed, names, eseq.data(), eoff);
  }
  if (!vcf.empty()) {
    const EditRecords er = fetch_edits(ctx, uint32_t(recs.size()));
    std::vector<std::string> names;
    std::vector<uint64_t> lens;
    for (size_t i = 0; i < recs.size(); i++) { names.push_back(recs[i].name); lens.push_back(off[i + 1] - off[i]); }
    write_edits_vcf(vcf, names, lens, &er);
  }
  gp_ctx_destroy(ctx);
  return 0;
}
