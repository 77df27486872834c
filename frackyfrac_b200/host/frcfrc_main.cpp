// C++ stand-in for the Go `frcfrc` binary (frcfrc/frcfrc.go): same flags, same
// validation and error behaviour, same stdout / -o bytes.  It exists because
// this image has no Go toolchain; INTEGRATION.md shows the cgo patch that makes
// the real Go main call the same C ABI.  The only thing replaced is the body
// of unifrac() (frcfrc.go:58): it now pulls ordered chunks from libfrcfrc_cuda.
#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "frcfrc_cuda.h"
#include "hostlib.hpp"

namespace {

const char* kUsage =
    "FrackyFrac calculates UniFrac on the given abundance table.\n"
    "Outputs one distance per line in the order (1,2),(1,3),(2,3)...(1,n)...(n-1,n).\n"
    "\n"
    "Params:\n";
// flag.PrintDefaults() layout for the flags of frcfrc.go:18-27 (sorted by name).
const char* kDefaults =
    "  -i string\n    \tPath to input file (default stdin)\n"
    "  -l\tLeave abundance values unnormalized (default normalize each sample to sum up to 1)\n"
    "  -o string\n    \tPath to output file (default stdout)\n"
    "  -p int\n    \tNumber of threads (default 1)\n"
    "  -s\tInput is in sparse format\n"
    "  -t string\n    \tPath to tree file, required\n"
    "  -w\tUse weighted UniFrac (default unweighted)\n";

[[noreturn]] void die(const std::string& msg) {  // common.ExitIfError (common/common.go:13-18)
  fprintf(stderr, "ERROR: %s\n", msg.c_str());
  exit(2);
}
void usage() { fputs(kUsage, stderr); fputs(kDefaults, stderr); }

struct Flags {
  std::string fin, fout, ftree;
  bool wgt = false, sparse = false, nnorm = false;
  long nt = 1;
};

bool parse_bool(const std::string& v, bool* out) {
  if (v == "1" || v == "t" || v == "T" || v == "true" || v == "TRUE" || v == "True") { *out = true; return true; }
  if (v == "0" || v == "f" || v == "F" || v == "false" || v == "FALSE" || v == "False") { *out = false; return true; }
  return false;
}

// Go's flag package: -x, --x, -x=v, -x v; parsing stops at the first non-flag or "--".
Flags parse_flags(int argc, char** argv) {
  Flags f;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a.size() < 2 || a[0] != '-') break;
    size_t d = a[1] == '-' ? 2 : 1;
    if (a.size() == 2 && d == 2) break;  // "--"
    std::string name = a.substr(d), val;
    bool has_val = false;
    size_t eq = name.find('=');
    if (eq != std::string::npos) { val = name.substr(eq + 1); name = name.substr(0, eq); has_val = true; }
    auto bad = [&](const std::string& m) { fprintf(stderr, "%s\n", m.c_str()); usage(); exit(2); };
    if (name == "h" || name == "help") { usage(); exit(0); }
    bool* bp = name == "w" ? &f.wgt : name == "s" ? &f.sparse : name == "l" ? &f.nnorm : nullptr;
    if (bp) {
      if (!has_val) *bp = true;
      else if (!parse_bool(val, bp)) bad("invalid boolean value \"" + val + "\" for -" + name + ": parse error");
      continue;
    }
    if (name != "i" && name != "o" && name != "t" && name != "p") bad("flag provided but not defined: -" + name);
    if (!has_val) {
      if (i + 1 >= argc) bad("flag needs an argument: -" + name);
      val = argv[++i];
    }
    if (name == "i") f.fin = val;
    else if (name == "o") f.fout = val;
    else if (name == "t") f.ftree = val;
    else {
      char* end = nullptr;
      errno = 0;
      f.nt = strtol(val.c_str(), &end, 0);
      if (val.empty() || *end || errno) bad("invalid value \"" + val + "\" for flag -p: parse error");
    }
  }
  return f;
}

}  // namespace

int main(int argc, char** argv) {
  if (argc == 1) { usage(); return 0; }  // frcfrc.go:71-74
  Flags fl = parse_flags(argc, argv);
  if (fl.ftree.empty()) die("please provide a tree file with -t");
  if (fl.nt < 1) die("bad number of threads: " + std::to_string(fl.nt));
  if (fl.nnorm && !fl.wgt) die("-l can only be used with weighted unifrac");

  auto t0 = std::chrono::steady_clock::now();
  const bool timing = getenv("FRC_CLI_TIMING") != nullptr;  // stage times on stderr (not part of the reference's output)
  auto tl = t0;
  auto lap = [&](const char* what) {
    if (!timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[timing] %-22s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - tl).count());
    tl = now;
  };
  double fmt_ms = 0, write_ms = 0, next_ms = 0;
  try {
    fputs("Reading tree\n", stderr);
    std::string tt = frchost::read_file(fl.ftree);
    frchost::FlatTree tree = frchost::parse_newick(tt.data(), tt.size());
    lap("read + parse tree");
    fputs("Loading abundances\n", stderr);
    std::string it = frchost::read_file(fl.fin);
    lap("read table file");
    frchost::Table tab = frchost::parse_table(it.data(), it.size(), fl.sparse, static_cast<int>(fl.nt));  // -p workers (frcfrc.go:42-50)
    lap("parse table");
    // FRCFRC_QUERY=<table> (stand-in only, like FRCFRC_PRUNE): -i is the reference table and the output is the
    // query x reference block, (q1,r1) ... (q1,rR), (q2,r1) ... (frc_create_cross); -s applies to both tables
    const char* fquery = getenv("FRCFRC_QUERY");
    frchost::Table qtab;
    if (fquery) {
      std::string qt = frchost::read_file(fquery);
      qtab = frchost::parse_table(qt.data(), qt.size(), fl.sparse, static_cast<int>(fl.nt));
      lap("read + parse query table");
    }
    fputs("Validating\n", stderr);
    frchost::Csr csr = frchost::resolve(tab, tree, static_cast<int>(fl.nt));
    frchost::Csr qcsr;
    if (fquery) qcsr = frchost::resolve(qtab, tree, static_cast<int>(fl.nt));
    lap("validate + resolve");

    frchost::Writer w(fl.fout, static_cast<int>(fl.nt));  // aio.Create (frcfrc.go:100-106): ".gz" / ".zst" by suffix

    fputs("Converting abundances\n", stderr);
    frc_tree_t ft{static_cast<int32_t>(tree.parent.size()), tree.parent.data(), tree.length.data()};
    frc_csr_t fc{tab.n_samples(), csr.row_ptr.data(), csr.col.data(), csr.val.data()};
    frc_csr_t fq{qtab.n_samples(), qcsr.row_ptr.data(), qcsr.col.data(), qcsr.val.data()};
    frc_opts_t fo{};
    fo.mode = fl.wgt ? FRC_WEIGHTED : FRC_UNWEIGHTED;
    // -l: the reference's behaviour as coded (normalize = 0: unifrac.go:108-110 skips the id-sort together with
    // the normalisation).  FRCFRC_L=documented selects what the flag's help text says (sorted lists, raw values).
    fo.normalize = fl.nnorm ? 0 : 1;
    if (fl.nnorm)
      if (const char* e = getenv("FRCFRC_L")) fo.normalize = !strcmp(e, "documented") ? 2 : 0;
    fo.path = FRC_PATH_AUTO;
    if (const char* e = getenv("FRCFRC_PATH")) fo.path = !strcmp(e, "exact") ? FRC_PATH_EXACT : !strcmp(e, "fast") ? FRC_PATH_FAST : FRC_PATH_AUTO;
    // -l as coded with FRCFRC_PATH=fast: the key-matched FP32 tiles (within 1e-5 of the reference, not bit-exact);
    // without FRCFRC_PATH, -l runs the bit-exact list walk
    if (fo.normalize == 0 && fo.path == FRC_PATH_FAST) fo.flags |= FRC_FLAG_L_TILES;
    // FRCFRC_PRUNE=1: run on the subtree the table observes (a large reference tree, a small table)
    if (const char* e = getenv("FRCFRC_PRUNE")) if (!strcmp(e, "1")) fo.flags |= FRC_FLAG_PRUNE;
    fo.device = -1;
    fo.world = 1;
    // every visible B200 works on the job; the engine hands their bands out as ONE ordered stream
    // (FRCFRC_DEVICES=n limits it to the first n; tiny inputs are not worth more than one context)
    fo.n_devices = -1;
    if (const char* e = getenv("FRCFRC_DEVICES")) fo.n_devices = std::max(1, atoi(e));
    else if (static_cast<double>(tab.n_samples()) * static_cast<double>(fquery ? qtab.n_samples() : tab.n_samples()) *
                 static_cast<double>(tree.parent.size()) < 4e12)
      fo.n_devices = 1;
    frc_job_t* job = nullptr;
    const int crc = fquery ? frc_create_cross(nullptr, &ft, &fc, &fq, &fo, &job) : frc_create(nullptr, &ft, &fc, &fo, &job);
    if (crc != FRC_OK) die(frc_last_error(nullptr));
    lap("frc_create (+ CUDA init)");
    fputs("Calculating distances\n", stderr);
    frc_info_t info;
    frc_job_info(job, &info);
    const bool f32 = info.value_bytes == 4;  // fast paths deliver fp32: format straight from the pinned ring
    std::vector<std::string> parts;  // one formatted piece per -p worker, written in order
    for (;;) {
      const double* d = nullptr; const float* f = nullptr; int64_t first, n;
      auto a0 = std::chrono::steady_clock::now();
      const int rc = f32 ? frc_next_f32(job, &f, &first, &n) : frc_next(job, &d, &first, &n);
      if (rc != FRC_OK) { std::string m = frc_last_error(job); frc_destroy(job); die(m); }
      if (n == 0) break;
      auto a1 = std::chrono::steady_clock::now();
      if (f32) {
        const int64_t* xi = nullptr; const double* xv = nullptr; int64_t nx = 0;
        frc_chunk_exceptions(job, &xi, &xv, &nx);
        frchost::format_parts_parallel_f32(f, n, first, xi, xv, nx, static_cast<int>(fl.nt), parts);
      } else {
        frchost::format_parts_parallel(d, n, static_cast<int>(fl.nt), parts);  // -p threads format, one writer
      }
      auto a2 = std::chrono::steady_clock::now();
      std::string werr;
      try {
        for (const std::string& p : parts) w.write(p.data(), p.size());
      } catch (const std::exception& e) { werr = e.what(); }
      auto a3 = std::chrono::steady_clock::now();
      next_ms += std::chrono::duration<double, std::milli>(a1 - a0).count();
      fmt_ms += std::chrono::duration<double, std::milli>(a2 - a1).count();
      write_ms += std::chrono::duration<double, std::milli>(a3 - a2).count();
      if (!werr.empty()) {  // frcfrc.go:59-63
        frc_destroy(job);
        die(werr);
      }
    }
    if (timing) fprintf(stderr, "[timing] frc_next waits %.1f ms, formatting %.1f ms, fwrite %.1f ms\n", next_ms, fmt_ms, write_ms);
    tl = std::chrono::steady_clock::now();
    frc_destroy(job);
    w.close();
    lap("destroy + close");
  } catch (const std::exception& e) {
    die(e.what());
  }
  double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  fprintf(stderr, "Took %.6gs\nDone\n", sec);
  return 0;
}
