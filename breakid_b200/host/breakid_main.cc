// breakid_main.cc -- drop-in `BreakID` command-line driver on top of the B200 C ABI.
//
// Same process contract as the reference main() (reference src/BreakID.cc:6-192): flags
// -i -o -n -q -t -fast -all -h -? (single-dash long options, src/BreakID.cc:15-26), outputs
// <o>_fusion.txt, <o>_fusion_all.txt (with -all), <o>_params.txt, <o>_performance.txt, error
// messages + exit(1) as the reference prints them (exit(-1), status 255, on its fatal "error cigar" path).  Differences, all additive and default-neutral:
//   * the option table is terminated, so unknown flags report an error instead of segfaulting, and
//     -t takes its argument (the reference declares has_arg=0 and then reads optarg);
//   * -s <k>   sd multiplier of the distance formula (the literal 3 at src/BreakID.cc:103);
//   * -r <refGene.txt> (default: $BREAKID_INSTALLDIR/ref_files/refGene.txt), -threads, -gpu;
//   * -gpu 0,1,2,...  several GPUs of one box: one host thread and one context per device, every rank inflates and
//     decodes its own BGZF block range of the BAM (genomic-bin sharding of the file itself), the exchanges between the
//     ranks are NCCL calls inside the library (bkid_dist_run).  A device may be named more than once (-gpu 0,0,0): the
//     ranks then share it and exchange through device copies -- that is how the path is tested on a one-GPU box;
//   * -sort  the BAM may be in any record order (e.g. read-name grouped, as bwa mem | samblaster writes it): the records are
//     coordinate sorted on the device after decode (bkid_sort_records), and no .bai is required.  One GPU only;
//   * -i may name SAM text instead of a BAM (a file whose first line is a header line or an alignment line of 11 or more
//     tab-separated fields), or be - to read SAM from stdin: the lines are parsed on the device (bkid_push_sam), and no
//     .bai is required.  A BAM (first bytes 1f 8b) takes the BAM path unchanged.  With -gpu a,b,... every rank parses
//     the newline-aligned byte range of a coordinate-sorted SAM file that falls to it; stdin needs one GPU.
// Host work: BAM / SAM header parsing (bam_reader.cc), .nib loading, refGene annotation, the final unstable sort
// by N_DRP and file writing.  Everything between decode and the cluster records runs on the GPU.
#include <getopt.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <set>
#include <string>
#include <thread>
#include <vector>

#include "../../include/breakid_b200.h"
#include "annotate.h"
#include "bam_reader.h"
#include "nibtools.h"

static const char *kHelp =
    " Usage: \n \t BreakID -i input.bam -o prefix -n nib_folder <options> \n\n "
    "     DESCRIPTION\n "
    "     \t -h -? -help \t help\n "
    "     \t -i*        \t input bam-file, or SAM text (a file, or - for stdin)\n "
    "     \t -o*        \t output file (prefix only)\n "
    "     \t -n*        \t folder name to nib files\n "
    "     \t -q         \t encompassing reads quality thresholds  [20]\n"
    "     \t -t         \t distance relative to (sqrt(2)*(insert size mean +3* insert size sd))  [2]\n "
    "     \t -fast      \t use the fast cluster strategy [default no] \n "
    "     \t -all       \t no filter enspan out [default is filter]  \n "
    "     \t -s         \t sd multiplier of the distance formula [3]\n "
    "     \t -r         \t refGene.txt [$BREAKID_INSTALLDIR/ref_files/refGene.txt]\n "
    "     \t -x         \t exclude regions (BED: chrom, start, end): records starting there are ignored [none]\n "
    "     \t -validate  \t split reads count only if their clipped bases align where the SA tag says (needs nib files) [off]\n "
    "     \t -threads   \t BAM decode threads [8]\n "
    "     \t -sort      \t input BAM in any record order: sort on the GPU, no index needed (one GPU only) [off]\n "
    "     \t -gpu       \t CUDA device, or a list / range such as 0,1 or 0-7 (one rank per entry, NCCL between them) [0]\n ";

static const char *kFusion[] = {"Unknown", "Translocation", "Inversion", "Duplication", "Deletion"};

struct CallRow {
  bkid_cluster_rec c;
  SideAnnotation a1, a2;
};

static bool exists(const std::string &p) { struct stat st; return stat(p.c_str(), &st) == 0; }
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// 0 = BAM (gzip magic), 1 = SAM (the first line is a header line or has at least 11 tab-separated fields), -1 = neither
static int sniff_input(const std::string &path)
{
  FILE *f = fopen(path.c_str(), "rb");
  if (!f) return -1;
  std::string b(65536, '\0');
  b.resize(fread(&b[0], 1, b.size(), f));
  fclose(f);
  if (b.size() >= 2 && (uint8_t)b[0] == 0x1f && (uint8_t)b[1] == 0x8b) return 0;
  if (b.empty()) return -1;
  if (b[0] == '@') return 1;
  std::string first = b.substr(0, b.find('\n'));
  return std::count(first.begin(), first.end(), '\t') >= 10 ? 1 : -1;
}

static bool cmp_cluster(const CallRow &a, const CallRow &b) { return a.c.n_discordant_pair > b.c.n_discordant_pair; }   // reference src/BreakID.h:185-188

static void write_header(std::ofstream &o)
{
  o << "Fusion_Type\tBreakPoint1\tBreakPoint2\tGene1\tBreakPoint_Info_Pair1\tGene2\tBreakPoint_Info_Pair2\tN_DRP\tN_SR\t"
       "BreakPoint1_Depth\tBreakPoint2_Depth\tBreakPoint1_AF\tBreakPoint2_AF\tBP1_Neighbour_Seq\tBP2_Neighbour_Seq\n";
}

static void write_row(std::ofstream &o, const CallRow &r, const std::vector<std::string> &names)
{
  auto nm = [&](int t) { return t >= 0 && t < (int)names.size() ? names[t] : std::string("*"); };
  const bkid_cluster_rec &c = r.c;
  o << kFusion[c.fusion_type] << "\t";
  o << nm(c.p1_tid) << ":" << c.p1_exact_pos << "\t";
  o << nm(c.p2_tid) << ":" << c.p2_exact_pos << "\t";
  o << r.a1.gene << "\t" << r.a1.strand << ":" << r.a1.exon_info << "\t";
  o << r.a2.gene << "\t" << r.a2.strand << ":" << r.a2.exon_info << "\t";
  o << (long)c.n_discordant_pair << "\t" << (long)c.n_split_read << "\t";
  o << c.p1_bp_depth << "\t" << c.p2_bp_depth << "\t";
  o << c.p1_alle_freq << "\t" << c.p2_alle_freq << "\t";
  o << c.p1_rpt << "\t" << c.p2_rpt << "\n";
}

// annotation, the final unstable sort by N_DRP and the four output files (reference src/BreakID.cc:492-567,1170-1263,175-191):
// shared by the single-GPU and the multi-GPU path.  `extra` writes the <o>_b200_timings.txt body.
template <typename Extra>
static void finish_and_write(const std::string &inp, const std::string &out, const std::string &refgene, const std::vector<std::string> &names,
                             const std::vector<bkid_cluster_rec> &cl, bool filter, bool need_index, int qual, double dist, bool reached_breakpoint_stage, double t_start,
                             int64_t n_pairs, int64_t n_masked, int64_t n_clustered, int64_t n_clusters, double t_scan, double t_cluster, double t_bp, Extra extra)
{
  std::vector<Transcript> tx;
  RefGeneIndex tx_index;
  std::vector<CallRow> rows;
  if (reached_breakpoint_stage) {
    // the reference opens the index and refGene as soon as one bucket reaches the break-point stage
    if (need_index && !exists(inp + ".bai") && !exists(inp.substr(0, inp.size() > 4 ? inp.size() - 4 : 0) + ".bai")) {
      std::cerr << "Error: please index bam-file first:\t" << inp << std::endl;                     // src/BreakID.cc:412-416
      exit(1);
    }
    if (!load_refgene(refgene, tx)) { std::cerr << "Error: cannot open \t" << refgene << std::endl; exit(1); }   // src/RefSeqTranscript.cc:205-209
    tx_index.build(tx);
    std::cout << "valid cluster count: " << cl.size() << std::endl;
    for (const bkid_cluster_rec &c : cl) {
      CallRow r;
      r.c = c;
      long p1 = (r.c.p1_exact_pos == (uint32_t)-1) ? (long)r.c.p1_mean_pos : (long)r.c.p1_exact_pos;   // src/BreakID.cc:518-534
      long p2 = (r.c.p2_exact_pos == -1) ? (long)r.c.p2_mean_pos : (long)r.c.p2_exact_pos;
      auto nm = [&](int t) { return t >= 0 && t < (int)names.size() ? names[t] : std::string("*"); };
      r.a1 = annotate_side(tx, tx_index, nm(r.c.p1_tid), p1);
      r.a2 = annotate_side(tx, tx_index, nm(r.c.p2_tid), p2);
      rows.push_back(r);
    }
  }
  // ---- write (src/BreakID.cc:1184-1263): unstable sort by N_DRP, same library sort on the same order ----
  std::sort(rows.begin(), rows.end(), cmp_cluster);
  std::ofstream o_all, o_f;
  if (!filter) { o_all.open((out + "_fusion_all.txt").c_str()); write_header(o_all); }
  o_f.open((out + "_fusion.txt").c_str());
  write_header(o_f);
  for (const CallRow &r : rows) {
    bool cond_all = r.c.n_split_read > 0 && r.c.p1_exact_pos != (uint32_t)-1 && r.c.p2_exact_pos != -1;
    bool cond_filter = cond_all && (!(r.a1.gene == "intergenic" && r.a2.gene == "intergenic") && r.a1.gene != r.a2.gene) && !r.c.is_rpt;
    if (cond_filter) write_row(o_f, r, names);
    if (!filter && cond_all) write_row(o_all, r, names);
  }
  if (!filter) o_all.close();
  o_f.close();
  {
    std::ofstream p((out + "_params.txt").c_str());                                                 // src/BreakID.cc:1170-1182
    p << "ENSPAN" << std::endl;
    p << "inp_file\t" << inp << std::endl;
    p << "out_file\t" << out << std::endl;
    p << "qual\t" << (long)qual << std::endl;
    p << "w\t" << dist << std::endl;
    p << "build\t" << "hg19" << std::endl;
  }
  double t_total = now_s() - t_start;
  std::cout << "the fusion process of file " << inp << "  costs time: " << t_total << " seconds" << std::endl;
  {
    std::ofstream p((out + "_performance.txt").c_str());                                            // src/BreakID.cc:175-191 (same columns, all filled)
    p << "scan_dist\tdiscordant pairs\tremove isolated\tafter_cluster\troot cluster\tscanning time\tcluster time\tfind breakpoint time\ttotal time" << std::endl;
    p << dist << "\t" << n_pairs << "\t" << n_masked << "\t" << n_clustered << "\t" << n_clusters << "\t" << t_scan << "\t" << t_cluster << "\t" << t_bp << "\t" << t_total
      << std::endl;
    std::ofstream j((out + "_b200_timings.txt").c_str());
    extra(j);
  }
}

int main(int argc, char *argv[])
{
  double t_start = now_s();
  static struct option longopts[] = {
      {"help", 0, 0, 'h'}, {"i", 1, 0, 1}, {"o", 1, 0, 2}, {"q", 1, 0, 3}, {"n", 1, 0, 4}, {"fast", 0, 0, 5}, {"t", 1, 0, 6},
      {"all", 0, 0, 7}, {"s", 1, 0, 8}, {"r", 1, 0, 9}, {"threads", 1, 0, 10}, {"gpu", 1, 0, 11}, {"x", 1, 0, 12}, {"validate", 0, 0, 13}, {"sort", 0, 0, 14}, {0, 0, 0, 0}};
  std::string inp, out, nib_dir, refgene, exclude_bed;
  int qual = 20, times = 2, sd_mult = 3, threads = 8, gpu = 0;
  std::vector<int> gpus;
  bool fast = false, filter = true, validate = false, sort = false;
  int opt, li;
  optind = 0;
  opterr = 0;
  while ((opt = getopt_long_only(argc, argv, "h?", longopts, &li)) != -1) {
    switch (opt) {
      case 'h': std::cerr << kHelp; exit(1);
      case 1: inp = optarg; break;
      case 2: out = optarg; break;
      case 3: qual = (int)labs(atol(optarg)); break;
      case 4: nib_dir = optarg; break;
      case 5: fast = true; break;
      case 6: times = (int)labs(atol(optarg)); break;
      case 7: filter = false; break;
      case 8: sd_mult = (int)labs(atol(optarg)); break;
      case 9: refgene = optarg; break;
      case 10: threads = std::max(1, atoi(optarg)); break;
      case 11: {
        gpus.clear();
        for (const char *q = optarg; *q;) {                 // "3", "0,1,2" or "0-7" (ranges and lists mix: "0-3,6")
          int a = atoi(q), b = a;
          while (*q && *q != ',' && *q != '-') ++q;
          if (*q == '-') { b = atoi(++q); while (*q && *q != ',') ++q; }
          if (b < a || b - a > 63) { std::cerr << "Error: bad -gpu range\n"; exit(1); }
          for (int g = a; g <= b; ++g) gpus.push_back(g);
          if (*q == ',') ++q;
        }
        gpu = gpus.empty() ? 0 : gpus[0];
        break;
      }
      case 12: exclude_bed = optarg; break;
      case 13: validate = true; break;
      case 14: sort = true; break;
      case '?':
        if (optopt == 0 && optind > 0 && (!strcmp(argv[optind - 1], "-?") || !strcmp(argv[optind - 1], "-help"))) { std::cerr << kHelp; exit(1); }
        std::cerr << kHelp;
        exit(1);
      default: std::cerr << "Error: cannot parse arguments.\n"; exit(1);
    }
  }
  if (inp.empty() || out.empty()) { std::cerr << kHelp; std::cerr << "Error: input- and output file is required.\n"; exit(1); }
  if (nib_dir.empty()) { std::cerr << kHelp; std::cerr << "Error: nib file's root dir is required.\n"; exit(1); }
  if (sort && gpus.size() > 1) {
    std::cerr << "Error: -sort works on one GPU only; sort the BAM first to use several (-gpu " << gpus.size() << " devices)\n";
    exit(1);
  }
  if (refgene.empty()) {
    const char *inst = getenv("BREAKID_INSTALLDIR");
    refgene = std::string(inst ? inst : ".") + "/ref_files/refGene.txt";
  }

  // ---- open: the host walks the BGZF block headers and parses the BAM header; inflate + record decode run on the
  // device (bkid_push_bgzf).  BKID_HOST_DECODE=1 selects the multi-threaded host decoder instead (A/B checks).
  std::cout << "start to stats the insert size...\n";
  char err[256];
  double t0 = now_s();
  const bool host_decode = getenv("BKID_HOST_DECODE") && atoi(getenv("BKID_HOST_DECODE")) != 0;
  bkid_host_bam *bam = nullptr;
  bkid_host_bgzf *bgzf = nullptr;
  bkid_host_sam *sam = nullptr;
  const bkid_header *hdr = nullptr;
  const bool from_stdin = inp == "-";
  const bool is_sam = from_stdin || sniff_input(inp) == 1;
  std::vector<uint8_t> sbuf;                           // stdin: the text read so far and not yet pushed
  size_t spos = 0;                                     // stdin: start of the unpushed text in sbuf
  bool seof = false;
  const size_t PIECE = (size_t)256 << 20;
  auto sfill = [&]() {
    size_t o = sbuf.size();
    sbuf.resize(o + PIECE);
    size_t n = fread(sbuf.data() + o, 1, PIECE, stdin);
    sbuf.resize(o + n);
    if (n == 0) seof = true;
  };
  if (is_sam && host_decode) { std::cerr << "Error: host decode reads BAM only (unset BKID_HOST_DECODE for SAM input)\n"; exit(1); }
  if (from_stdin && gpus.size() > 1) { std::cerr << "Error: SAM from stdin needs one GPU; give a SAM file to use several (-gpu " << gpus.size() << " devices)\n"; exit(1); }
  if (from_stdin) {
    for (;;) {                                         // the header lines come first
      if (spos >= sbuf.size()) { if (seof) break; sfill(); continue; }
      if (sbuf[spos] != '@') break;
      const void *nl = memchr(sbuf.data() + spos, '\n', sbuf.size() - spos);
      if (!nl) { if (seof) { spos = sbuf.size(); break; } sfill(); continue; }
      spos = (size_t)((const uint8_t *)nl - sbuf.data()) + 1;
    }
    sam = bkid_host_sam_parse(sbuf.data(), spos, err, sizeof err);
    if (!sam) { std::cerr << "Error: can not read sam header from stdin: " << err << std::endl; exit(1); }
    hdr = bkid_host_sam_header(sam);
  } else if (is_sam) {
    sam = bkid_host_sam_open(inp.c_str(), err, sizeof err);
    if (!sam) { std::cerr << "Error: can not open sam-file: " << inp << " (" << err << ")" << std::endl; exit(1); }
    hdr = bkid_host_sam_header(sam);
  } else if (host_decode) {
    bam = bkid_host_read_bam(inp.c_str(), threads, err, sizeof err);
    if (!bam) { std::cerr << "Error: can not open bam-file: " << inp << std::endl; exit(1); }
    hdr = bkid_host_bam_header(bam);
  } else {
    bgzf = bkid_host_bgzf_open(inp.c_str(), err, sizeof err);
    if (!bgzf) { std::cerr << "Error: can not open bam-file: " << inp << std::endl; exit(1); }
    hdr = bkid_host_bgzf_header(bgzf);
  }
  double t_decode = now_s() - t0;
  {
    std::ifstream in((nib_dir + "/ref_names.txt").c_str());
    if (!in.is_open()) { std::cerr << "Error: cannot open reference names file.\n"; exit(1); }     // src/BreakID.cc:1399-1404
  }
  std::vector<std::string> names;
  for (int i = 0; i < hdr->n_targets; ++i) names.emplace_back(hdr->target_name[i]);

  // ---- device ----
  bkid_params prm;
  bkid_default_params(&prm);
  prm.qual = qual; prm.times = times; prm.fast = fast ? 1 : 0; prm.sd_mult = sd_mult; prm.validate_align = validate ? 1 : 0;
  std::vector<int32_t> xt, xb, xe;
  if (!exclude_bed.empty()) {                          // additive: -x regions.bed (chrom, 0-based start, end); not a reference flag
    std::ifstream bed(exclude_bed.c_str());
    if (!bed.is_open()) { std::cerr << "Error: cannot open exclude bed-file: " << exclude_bed << std::endl; exit(1); }
    std::string line;
    while (std::getline(bed, line)) {
      if (line.empty() || line[0] == '#' || !line.compare(0, 5, "track") || !line.compare(0, 7, "browser")) continue;
      char chrom[256]; long b = 0, e = 0;
      if (sscanf(line.c_str(), "%255s %ld %ld", chrom, &b, &e) != 3) continue;
      for (int t = 0; t < hdr->n_targets; ++t)
        if (names[t] == chrom) { xt.push_back(t); xb.push_back((int32_t)b); xe.push_back((int32_t)e); break; }
    }
  }
  const int W = (int)std::max<size_t>(gpus.size(), 1);
  if (W > 1) {
    // ================= several GPUs: one rank per -gpu entry, sharded ingest, exchanges inside the library =================
    if (host_decode) { std::cerr << "Error: -gpu with several devices needs the device decoder (unset BKID_HOST_DECODE)\n"; exit(1); }
    std::vector<bkid_ctx *> ctxs(W, nullptr);
    for (int r = 0; r < W; ++r) {
      ctxs[r] = bkid_create(gpus[r], hdr, &prm);
      if (!ctxs[r]) { std::cerr << "Error: " << bkid_last_error(nullptr) << std::endl; exit(1); }
      if (!xt.empty() && bkid_set_exclude(ctxs[r], (int64_t)xt.size(), xt.data(), xb.data(), xe.data())) { std::cerr << "Error: set_exclude: " << bkid_last_error(ctxs[r]) << std::endl; exit(1); }
    }
    double t_push0 = now_s();
    std::vector<int64_t> nrec(W, 0);
    std::vector<uint64_t> first(W, 0), next(W, 0);
    std::vector<int> rcs(W, 0);
    if (sam) {
      // rank r parses the newline-aligned byte range [cut_r, cut_r+1): cut_r is the first line start at or after r * size / W
      const uint8_t *text = bkid_host_sam_data(sam);
      const uint64_t size = bkid_host_sam_size(sam), f0 = bkid_host_sam_first_record(sam);
      std::vector<uint64_t> cut(W + 1, size);
      cut[0] = f0;
      for (int r = 1; r < W; ++r) {
        uint64_t p = std::max<uint64_t>(f0, size * (uint64_t)r / (uint64_t)W);
        if (p > f0 && p < size && text[p - 1] != '\n') {
          const void *nl = memchr(text + p, '\n', (size_t)(size - p));
          p = nl ? (uint64_t)((const uint8_t *)nl - text) + 1 : size;
        }
        cut[r] = std::max(p, cut[r - 1]);
      }
      std::vector<int64_t> lines(W + 1, bkid_host_sam_first_line(sam));     // file line number of every cut (error messages)
      {
        std::vector<std::thread> th;
        for (int r = 0; r < W; ++r) th.emplace_back([&, r] { lines[r + 1] = std::count(text + cut[r], text + cut[r + 1], '\n'); });
        for (auto &t : th) t.join();
        for (int r = 0; r < W; ++r) lines[r + 1] += lines[r];
      }
      std::vector<std::thread> th;
      for (int r = 0; r < W; ++r)
        th.emplace_back([&, r] { rcs[r] = bkid_push_sam(ctxs[r], text + cut[r], cut[r + 1] - cut[r], lines[r], &nrec[r]); });
      for (auto &t : th) t.join();
      for (int r = 0; r < W; ++r)
        if (rcs[r]) { std::cerr << "Error: can not read sam-file: " << inp << " (" << bkid_last_error(ctxs[r]) << ")" << std::endl; exit(1); }
    } else {
    const int64_t nblk = bkid_host_bgzf_n_blocks(bgzf);
    {
      std::vector<std::thread> th;
      for (int r = 0; r < W; ++r)
        th.emplace_back([&, r] {
          rcs[r] = bkid_push_bgzf_range(ctxs[r], bkid_host_bgzf_data(bgzf), bkid_host_bgzf_size(bgzf), bkid_host_bgzf_blocks(bgzf), nblk, bkid_host_bgzf_first_record(bgzf),
                                        nblk * r / W, nblk * (r + 1) / W, &nrec[r], &first[r], &next[r]);
        });
      for (auto &t : th) t.join();
    }
    for (int r = 0; r < W; ++r)
      if (rcs[r]) { std::cerr << "Error: can not read bam-file: " << inp << " (" << bkid_last_error(ctxs[r]) << ")" << std::endl; exit(1); }
    for (int r = 0; r + 1 < W; ++r)        // where one range landed is where the next one started: the union is exactly the file's record sequence
      if (next[r] != first[r + 1]) { std::cerr << "Error: can not read bam-file: " << inp << " (the block ranges of ranks " << r << " and " << r + 1 << " do not stitch)" << std::endl; exit(1); }
    }
    double t_push = now_s() - t_push0;
    // nib files are needed by the refinement of every rank (41-mers are replicated work)
    for (int t = 0; t < hdr->n_targets; ++t) {
      nib nb;
      if (nb.open(nib_dir + "/hg19_" + names[t] + ".nib") == 0)
        for (int r = 0; r < W; ++r)
          if (bkid_set_nib(ctxs[r], t, nb.payload(), nb.size())) { std::cerr << "Error: set_nib: " << bkid_last_error(ctxs[r]) << std::endl; exit(1); }
    }
    std::vector<bkid_comm *> comms(W, nullptr);
    const bool distinct = std::set<int>(gpus.begin(), gpus.end()).size() == (size_t)W;
    if ((distinct ? bkid_comm_nccl_init_all(gpus.data(), W, comms.data()) : bkid_comm_local_create(W, comms.data())) != 0) {
      std::cerr << "Error: cannot create the communicators: " << bkid_last_error(nullptr) << std::endl; exit(1);
    }
    std::vector<double> mean(W), sd(W), dist(W);
    std::vector<int64_t> ncall(W);
    double t_run0 = now_s();
    std::cout << "Scanning discordant read pairs ...\n";
    if (int rc = bkid_dist_run_threads(ctxs.data(), comms.data(), W, fast ? 1 : 0, mean.data(), sd.data(), dist.data(), ncall.data())) {
      for (int r = 0; r < W; ++r) if (*bkid_last_error(ctxs[r])) std::cerr << "Error: rank " << r << ": " << bkid_last_error(ctxs[r]) << std::endl;
      exit(rc == BKID_ERR_CIGAR ? -1 : 1);
    }
    std::cout << "Scanning discordant read pairs done.\n";
    double t_run = now_s() - t_run0;
    std::cout << "the insert size mean: " << mean[0] << ", the insert size sd:" << sd[0] << " .\n";
    std::cout << "cluster_dist = span_dist = mask_dist = scan_dist = " << dist[0] << " .\n";
    std::vector<bkid_cluster_rec> cl((size_t)std::max<int64_t>(ncall[0], 1));
    int64_t n = 0;
    if (bkid_fetch_clusters(ctxs[0], cl.data(), (int64_t)cl.size(), &n)) { std::cerr << "Error: fetch_clusters: " << bkid_last_error(ctxs[0]) << std::endl; exit(1); }
    cl.resize((size_t)n);
    int64_t pairs = 0, masked = 0, clustered = 0, nclusters = 0, records = 0;
    for (int r = 0; r < W; ++r) { bkid_timings t; bkid_get_timings(ctxs[r], &t); pairs += t.n_pairs; masked += t.n_masked; clustered += t.n_clustered; nclusters += t.n_clusters; records += nrec[r]; }
    finish_and_write(inp, out, refgene, names, cl, filter, !sam, qual, dist[0], clustered > 0, t_start, pairs, masked, clustered, nclusters, t_run, 0.0, 0.0,
                     [&](std::ofstream &j) { j << "decoder\t" << (sam ? "sam" : "device") << "\nranks\t" << W << "\ncommunicator\t" << (distinct ? "nccl" : "local") << "\nopen_s\t" << t_decode << "\npush_s\t" << t_push
                                                << "\nrun_s\t" << t_run << "\nrecords\t" << records << "\n"; });
    for (int r = 0; r < W; ++r) { bkid_comm_destroy(comms[r]); bkid_destroy(ctxs[r]); }
    if (bgzf) bkid_host_bgzf_close(bgzf);
    if (sam) bkid_host_sam_close(sam);
    return 0;
  }
  bkid_ctx *ctx = bkid_create(gpu, hdr, &prm);
  if (!ctx) { std::cerr << "Error: " << bkid_last_error(nullptr) << std::endl; exit(1); }
  auto die = [&](const char *what) { std::cerr << "Error: " << what << ": " << bkid_last_error(ctx) << std::endl; exit(1); };
  if (!xt.empty() && bkid_set_exclude(ctx, (int64_t)xt.size(), xt.data(), xb.data(), xe.data())) die("set_exclude");
  double t_push0 = now_s();
  bkid_decode_stats dst;
  memset(&dst, 0, sizeof dst);
  if (host_decode) {
    if (bkid_push_batch(ctx, bkid_host_bam_batch_narrow(bam))) die("push_batch");
  } else if (sam) {
    auto push = [&](const uint8_t *text, uint64_t len, int64_t line) -> int64_t {
      int64_t nrec = 0;
      if (bkid_push_sam(ctx, text, len, line, &nrec)) {
        std::cerr << "Error: can not read sam-file: " << inp << " (" << bkid_last_error(ctx) << ")" << std::endl;
        exit(1);
      }
      bkid_decode_stats s;
      bkid_get_decode_stats(ctx, &s);
      dst.n_chunks += s.n_chunks; dst.uncompressed_bytes += s.uncompressed_bytes; dst.n_records += s.n_records;
      dst.total_ms += s.total_ms; dst.boundaries_ms += s.boundaries_ms; dst.extract_ms += s.extract_ms;
      return nrec;
    };
    int64_t line = bkid_host_sam_first_line(sam);
    if (!from_stdin) {
      const uint64_t f0 = bkid_host_sam_first_record(sam);
      push(bkid_host_sam_data(sam) + f0, bkid_host_sam_size(sam) - f0, line);
    } else {
      for (;;) {                                       // each call gets the complete lines read so far; a partial last line waits
        const bool last = seof;
        size_t end = sbuf.size();
        if (!last) {
          const void *nl = spos < sbuf.size() ? memrchr(sbuf.data() + spos, '\n', sbuf.size() - spos) : nullptr;
          end = nl ? (size_t)((const uint8_t *)nl - sbuf.data()) + 1 : spos;
        }
        if (end > spos) line += push(sbuf.data() + spos, end - spos, line);
        if (last) break;
        sbuf.erase(sbuf.begin(), sbuf.begin() + end);
        spos = 0;
        sfill();
      }
    }
  } else {
    int64_t nrec = 0;
    if (bkid_push_bgzf(ctx, bkid_host_bgzf_data(bgzf), bkid_host_bgzf_size(bgzf), bkid_host_bgzf_blocks(bgzf), bkid_host_bgzf_n_blocks(bgzf), bkid_host_bgzf_first_record(bgzf), &nrec)) {
      std::cerr << "Error: can not read bam-file: " << inp << " (" << bkid_last_error(ctx) << ")" << std::endl;
      exit(1);
    }
    bkid_get_decode_stats(ctx, &dst);
  }
  double t_push = now_s() - t_push0;
  double t_sort = 0;
  int32_t was_sorted = 1;
  if (sort) {
    double t1 = now_s();
    if (bkid_sort_records(ctx, &was_sorted)) die("sort_records");
    t_sort = now_s() - t1;
  }
  double mean = 0, sd = 0;
  if (bkid_insert_stats(ctx, &mean, &sd)) die("insert_stats");
  std::cout << "the insert size mean: " << mean << ", the insert size sd:" << sd << " .\n";
  double dist = times * sqrt((double)times) * (mean + sd_mult * sd);                                 // src/BreakID.cc:103
  std::cout << "cluster_dist = span_dist = mask_dist = scan_dist = " << dist << " .\n";
  double t_scan0 = now_s();
  int64_t n_pairs = 0, n_clusters = 0, n_called = 0;
  std::cout << "Scanning discordant read pairs ...\n";
  if (bkid_scan(ctx, dist, &n_pairs)) die("scan");
  std::cout << "Scanning discordant read pairs done.\n";
  double t_scan = now_s() - t_scan0;
  double t_cl0 = now_s();
  if (bkid_cluster(ctx, dist, fast ? 1 : 0, &n_clusters)) die("cluster");
  double t_cluster = now_s() - t_cl0;
  bkid_timings tm;
  bkid_get_timings(ctx, &tm);
  std::vector<bkid_cluster_rec> cl;
  double t_bp = 0;
  if (tm.n_clustered > 0) {
    if (!sort && !sam && !exists(inp + ".bai") && !exists(inp.substr(0, inp.size() > 4 ? inp.size() - 4 : 0) + ".bai")) {
      std::cerr << "Error: please index bam-file first:\t" << inp << std::endl;                     // src/BreakID.cc:412-416
      exit(1);
    }
    for (int t = 0; t < hdr->n_targets; ++t) {
      nib nb;
      if (nb.open(nib_dir + "/hg19_" + names[t] + ".nib") == 0)                                     // src/util_bam.cc:83-86
        if (bkid_set_nib(ctx, t, nb.payload(), nb.size())) die("set_nib");
    }
    double t1 = now_s();
    if (int rc = bkid_refine(ctx, dist, &n_called)) {
      std::cerr << "Error: refine: " << bkid_last_error(ctx) << std::endl;
      exit(rc == BKID_ERR_CIGAR ? -1 : 1);                                                           // the reference's exit(-1), src/BreakID.cc:954-968
    }
    t_bp = now_s() - t1;
    cl.resize((size_t)std::max<int64_t>(n_called, 1));
    int64_t n = 0;
    if (bkid_fetch_clusters(ctx, cl.data(), (int64_t)cl.size(), &n)) die("fetch_clusters");
    cl.resize((size_t)n);
  }
  bkid_get_timings(ctx, &tm);
  finish_and_write(inp, out, refgene, names, cl, filter, !sort && !sam, qual, dist, tm.n_clustered > 0, t_start, n_pairs, tm.n_masked, tm.n_clustered, n_clusters, t_scan, t_cluster, t_bp,
                   [&](std::ofstream &j) {
                     if (sam)
                       j << "decoder\tsam\nopen_s\t" << t_decode << "\npush_s\t" << t_push << "\ntext_bytes\t" << dst.uncompressed_bytes << "\nlines_ms\t" << dst.boundaries_ms << "\nparse_ms\t" << dst.extract_ms
                         << "\nsam_chunks\t" << dst.n_chunks;
                     else
                       j << "decoder\t" << (host_decode ? "host" : "device") << "\nopen_s\t" << t_decode << "\npush_s\t" << t_push << "\ninflate_ms\t" << dst.inflate_ms << "\nboundaries_ms\t" << dst.boundaries_ms
                         << "\nextract_ms\t" << dst.extract_ms << "\ncompressed_bytes\t" << dst.compressed_bytes << "\nuncompressed_bytes\t" << dst.uncompressed_bytes;
                     j << "\nrecords\t" << tm.n_records << "\nh2d_ms\t" << tm.h2d << "\nclassify_ms\t" << tm.classify << "\ninsert_stats_ms\t" << tm.insert_stats
                       << "\njoin_ms\t" << tm.join << "\nbucket_sort_ms\t" << tm.bucket_sort << "\nmask_ms\t" << tm.mask << "\ncluster_ms\t" << tm.cluster << "\nsummarize_ms\t" << tm.summarize
                       << "\nevidence_ms\t" << tm.evidence << "\nrefine_ms\t" << tm.refine << "\n";
                     if (sort) j << "sort_ms\t" << t_sort * 1e3 << "\ninput_was_sorted\t" << was_sorted << "\n";
                   });
  bkid_destroy(ctx);
  if (bam) bkid_host_bam_free(bam);
  if (bgzf) bkid_host_bgzf_close(bgzf);
  if (sam) bkid_host_sam_close(sam);
  return 0;
}
