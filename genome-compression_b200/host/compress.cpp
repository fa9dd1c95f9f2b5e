// compress.cpp — host driver of the B200 shared_tree path.
//
// Same command line as the reference's compress.cpp (flags at compress.cpp:82-93 of the
// reference: --help --verbose --statistics --no-save --output= --histogram= --dna-size=) and
// the same --statistics CSV line, extended with device throughput; plus --decompress, which
// the reference lacks (its .dag format does not record dna::size, so it must be given).
// Everything below the flag parsing is calls into the shim in include/ (one C-ABI call each).
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "shared_tree.h"

namespace fs = std::filesystem;
using clk = std::chrono::steady_clock;

struct Options {
  fs::path input, output, histogram, regions;
  bool verbose = false, statistics = false, save = true, decompress = false;
  std::size_t dna_size = 12;
};

static void usage() {
  std::cout << "Usage: compress_b200 [options] file\n"
               "  --help               this text\n"
               "  --verbose            human-readable report\n"
               "  --statistics         one CSV line: dna_size,width,ratio,in_bytes,out_bytes,construct_ms,sort_ms,total_ms,build_gbp_s\n"
               "  --no-save            do not write the .dag file\n"
               "  --output=<file>      output path (default <input>.dag, or <input>.txt with --decompress)\n"
               "  --histogram=<file>   write per-layer reference-count histograms (CSV)\n"
               "  --dna-size=<n>       nucleotides per leaf, 1..16 (default 12)\n"
               "  --decompress         input is a .dag file; write the decoded sequence as text\n"
               "  --regions=<file>     with --decompress: write only the regions of a BED file (chrom start end\n"
               "                       [name [score [strand]]], 0-based half-open; strand '-' = reverse complement)\n"
               "                       as FASTA, one record per region in file order (default output <input>.fa)\n";
}

static Options parse(int argc, char** argv) {
  Options o;
  for (int i = 1; i < argc; ++i) {
    const std::string a = argv[i];
    auto value = [&](const char* key) { return a.substr(std::strlen(key)); };
    if (a == "--help") { usage(); std::exit(0); }
    else if (a == "--verbose") o.verbose = true;
    else if (a == "--statistics") o.statistics = true;
    else if (a == "--no-save") o.save = false;
    else if (a == "--decompress") o.decompress = true;
    else if (a.rfind("--output=", 0) == 0) o.output = value("--output=");
    else if (a.rfind("--histogram=", 0) == 0) o.histogram = value("--histogram=");
    else if (a.rfind("--regions=", 0) == 0) o.regions = value("--regions=");
    else if (a.rfind("--dna-size=", 0) == 0) o.dna_size = (std::size_t)std::atoi(value("--dna-size=").c_str());
    else if (o.input.empty()) o.input = a;
    else { std::cout << "Compression of multiple files at once is currently not supported.\n"; std::exit(1); }
  }
  if (o.verbose && o.statistics) { std::cout << "Invalid flag combination: --verbose and --statistics are mutually exclusive\n"; std::exit(2); }
  if (o.input.empty()) { std::cout << "Invalid command: argument <file> required.\nUse --help for more information\n"; std::exit(2); }
  if (o.dna_size < 1 || o.dna_size > 16) { std::cout << "Invalid --dna-size: 1..16 supported\n"; std::exit(2); }
  if (!fs::is_regular_file(o.input)) { std::cout << "Invalid filename: " << o.input << '\n'; std::exit(2); }
  if (!o.regions.empty() && !o.decompress) { std::cout << "Invalid flag combination: --regions needs --decompress\n"; std::exit(2); }
  if (o.output.empty() && o.save) {
    o.output = o.input;
    o.output.replace_extension(!o.decompress ? ".dag" : o.regions.empty() ? ".txt" : ".fa");
  }
  return o;
}

static double ms_since(clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); }

struct Region {
  std::string chrom;
  uint64_t start = 0, end = 0;
  uint8_t strand = 0;
  std::size_t line = 0;
};

static bool parse_u64(const std::string& s, uint64_t& v) {
  if (s.empty() || s.size() > 19 || s.find_first_not_of("0123456789") != std::string::npos) return false;
  v = std::stoull(s);
  return true;
}

[[noreturn]] static void bed_error(std::size_t line, const std::string& what) {
  std::cerr << "line " << line << ": " << what << '\n';
  std::exit(1);
}

// BED: whitespace-separated `chrom start end [name [score [strand]]]`; empty lines and lines starting with
// '#', "track" or "browser" are skipped.  Any malformed line ends the program before the device is touched.
static std::vector<Region> read_bed(const fs::path& path) {
  std::ifstream in{path};
  if (!in) { std::cerr << "cannot read " << path << '\n'; std::exit(1); }
  std::vector<Region> regions;
  std::string text;
  for (std::size_t line = 1; std::getline(in, text); ++line) {
    std::istringstream fields{text};
    std::vector<std::string> f;
    for (std::string w; fields >> w;) f.push_back(w);
    if (f.empty() || f[0][0] == '#' || f[0] == "track" || f[0] == "browser") continue;
    if (f.size() < 3) bed_error(line, "expected chrom, start and end");
    Region r;
    r.chrom = f[0];
    r.line = line;
    if (!parse_u64(f[1], r.start)) bed_error(line, "start is not a non-negative integer: " + f[1]);
    if (!parse_u64(f[2], r.end)) bed_error(line, "end is not a non-negative integer: " + f[2]);
    if (r.start > r.end) bed_error(line, "start " + f[1] + " > end " + f[2]);
    if (f.size() >= 6) {
      if (f[5] == "-") r.strand = 1;
      else if (f[5] != "+" && f[5] != ".") bed_error(line, "strand is not '+', '-' or '.': " + f[5]);
    }
    regions.push_back(r);
  }
  return regions;
}

// One stb_extract_regions call for every region of the BED file, written as FASTA records.
static int extract(const Options& o) {
  const std::vector<Region> regions = read_bed(o.regions);
  std::ifstream in{o.input, std::ios::binary};
  shared_tree tree = shared_tree::deserialize(in);
  const uint64_t bases = (uint64_t)tree.width() * dna::size();
  std::vector<uint64_t> start(regions.size()), end(regions.size());
  std::vector<uint8_t> strand(regions.size());
  uint64_t total = 0;
  for (std::size_t i = 0; i < regions.size(); ++i) {
    const Region& r = regions[i];
    if (r.end > bases) bed_error(r.line, "end " + std::to_string(r.end) + " is past the sequence (" + std::to_string(bases) + " bases)");
    start[i] = r.start;
    end[i] = r.end;
    strand[i] = r.strand;
    total += r.end - r.start;
  }
  std::string seq(total, '\0');
  uint64_t written = 0;
  const int st = stb_extract_regions(tree.handle(), start.data(), end.data(), strand.data(), regions.size(), seq.data(),
                                     seq.size(), STB_HOST, &written);
  if (st != STB_OK) { std::cerr << stb_last_error(tree.handle()) << '\n'; return 1; }
  if (o.save) {
    std::ofstream out{o.output, std::ios::binary};
    uint64_t at = 0;
    for (const Region& r : regions) {
      out << '>' << r.chrom << ':' << r.start << '-' << r.end << '(' << (r.strand ? '-' : '+') << ")\n";
      out.write(seq.data() + at, (std::streamsize)(r.end - r.start)) << '\n';
      at += r.end - r.start;
    }
  }
  if (o.verbose || o.statistics) std::cout << dna::size() << ',' << regions.size() << ',' << written << '\n';
  return 0;
}

static int decompress(const Options& o) {
  if (!o.regions.empty()) return extract(o);
  std::ifstream in{o.input, std::ios::binary};
  shared_tree tree = shared_tree::deserialize(in);
  const std::size_t width = tree.width();
  std::string text(width * dna::size(), '\0');
  const int st = stb_decode_ascii(tree.handle(), 0, width, text.data(), STB_HOST);
  if (st != STB_OK) { std::cerr << stb_last_error(tree.handle()) << '\n'; return 1; }
  if (o.save) std::ofstream{o.output, std::ios::binary}.write(text.data(), (std::streamsize)text.size());
  if (o.verbose || o.statistics) std::cout << dna::size() << ',' << width << ',' << text.size() << '\n';
  return 0;
}

int main(int argc, char** argv) {
  const Options o = parse(argc, argv);
  dna::size(o.dna_size);
  if (o.decompress) return decompress(o);
  const auto in_bytes = fs::file_size(o.input);
  if (o.verbose) std::cout << " Filename: " << o.input << "\n Size:     " << bytes_to_string(in_bytes) << "\n";

  auto t0 = clk::now();
  shared_tree tree{o.input, o.verbose};
  const double construct_ms = ms_since(t0);
  t0 = clk::now();
  tree.sort_tree(o.verbose);
  const double sort_ms = ms_since(t0);

  const std::size_t out_bytes = tree.bytes(), width = tree.width();
  if (!o.histogram.empty()) tree.store_histogram(o.histogram);
  if (!o.output.empty() && o.save) tree.save(o.output);

  const double gbps = double(width * dna::size()) / (construct_ms * 1e6);
  if (o.verbose) {
    std::cout << " Output:            " << o.output << "\n Size:              " << bytes_to_string(out_bytes)
              << "\n Nucleotides:       " << width * dna::size() << "\n Compression ratio: " << double(in_bytes) / double(out_bytes)
              << "\n Leaf size:         " << dna::size() << "\n Width:             " << width << "\n Depth:             " << tree.depth()
              << "\n Leaves:            " << tree.leaf_count() << "\n Nodes:             " << tree.node_count()
              << "\n Tree construction: " << construct_ms << " ms (" << gbps << " Gbp/s incl. file read + H2D)\n Frequency sorting: " << sort_ms << " ms\n";
  }
  if (o.statistics)
    std::cout << dna::size() << ',' << width << ',' << double(in_bytes) / double(out_bytes) << ',' << in_bytes << ',' << out_bytes << ','
              << (long long)construct_ms << ',' << (long long)sort_ms << ',' << (long long)(construct_ms + sort_ms) << ',' << gbps << '\n';
  return 0;
}
