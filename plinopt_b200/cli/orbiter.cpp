// bin/orbiter -- drop-in for src/orbiter.cpp:365-441: random DeGroote-orbit search writing
// <stem>.nnz.sms next to every input when the winner improves on it (:338-348).
// Flags of the reference are kept; -P "X^2-d" searches over Q(sqrt d) (entries a + bX), while -z/-c
// (SLP-operation and canonical measures), -I and other polynomials are out of scope and rejected.
// Added: -g (minimise the growth factor G2 instead of the sparsity), --seed N, --exhaustive, --any-shape.
#include <cstdlib>

#include "cli_common.hpp"

static void usage(const char* prg, size_t loops) {
  std::clog << "Usage: " << prg << "  [-h|-O/-b #|-m/-q #|-r # # #|-P \"X^2-d\"|-s|-g] L.sms R.sms P.sms\n"
            << "  [-b b]: random check with values of size 'bitsize' (at most 32 here)\n"
            << "  [-m/-q m]: check is modulo (mod) or (mod/2^k) (default no)\n"
            << "  [-r r e s]: check is modulo (r^e-s) or ((r^e-s)/2^k) (default no)\n"
            << "  [-P \"X^2-d\"]: entries a+bX in Q(sqrt d), X^2 = d (default no)\n"
            << "  [-s|-g]: search sparser|lower growth factor (default is sparser)\n"
            << "  [-O #]: randomized search with that many loops (default " << loops << " loops)\n"
            << "  [--seed #] [--exhaustive]: candidate enumeration (default Philox, seed 0x504C494E4F505431)\n"
            << "  [--gpus #]: shard the sweep over that many GPUs of this box (default 1)\n"
            << "  [--any-shape]: run shapes without a compiled kernel on the runtime-shape kernels (any m, k, n <= 8)\n";
  exit(-1);
}

static void verdict_line(int v, int m, int k, int n, uint32_t nnz, uint32_t nno) {
  if (v == 0) std::clog << "# \033[1;32mSUCCESS: correct " << m << 'x' << k << 'x' << n << " {" << nnz << ',' << nno << "} Matrix-Multiplication \033[0m" << std::endl;
  else std::cerr << "# \033[1;31m****** ERROR, not a " << m << 'x' << k << 'x' << n << " MM algorithm******\033[0m" << std::endl;
}
// '# Found opt:' lines of src/orbiter.cpp:312-315, in index order (deterministic)
static void found_lines(const plo_orbiter_report& rep, const std::vector<plo_orbit_best>& recs, uint64_t nrec) {
  double bestopt = rep.init_score;
  uint32_t bnnz = rep.init_nnz, bnno = rep.init_nno;
  for (uint64_t t = 0; t < nrec; ++t) {
    std::clog << "# Found opt: " << recs[t].score << (recs[t].score < bestopt ? '<' : '=') << bestopt << "\t{" << recs[t].nnz << ',' << recs[t].nno << "}&{" << bnnz << ','
              << bnno << "}\t[" << recs[t].index << "/gpu]" << std::endl;
    bestopt = recs[t].score; bnnz = recs[t].nnz; bnno = recs[t].nno;
  }
}
static void reduced_line(const plo_orbiter_report& rep) {
  std::clog << "# \033[1;36mRdcd. opt: " << rep.best.score << '<' << rep.init_score << "\t{" << rep.best.nnz << ',' << rep.best.nno << "}\033[0m\t[" << rep.best.index << ']' << std::endl;
}

int main(int argc, char** argv) {
  unsigned long long loops = 100, seed = 0x504C494E4F505431ull;  // DEFAULT_RANDOM_LOOPS, plinopt_library.h:37-39
  int measure = PLO_MEASURE_NNZ, mode = PLO_MODE_PHILOX;
  cli::CheckFlags flags;
  std::vector<std::string> files;
  for (int i = 1; i < argc; ++i) {
    const std::string a(argv[i]);
    if (a == "--seed" && i + 1 < argc) seed = strtoull(argv[++i], nullptr, 0);
    else if (a == "--gpus" && i + 1 < argc) plo_set_sweep_devices(atoi(argv[++i]));
    else if (a == "--exhaustive") mode = PLO_MODE_EXHAUSTIVE;
    else if (a == "--any-shape") plo_set_orbit_any_shape(1);
    else if (a[0] == '-' && a.size() > 1) {
      if (a[1] == 'h') usage(argv[0], loops);
      else if (const int t = flags.take(argc, argv, i)) {
        if (t < 0) return -1;
        // -b is the bit size of the random integer inputs of the reference's over-Q check (plinopt_library.inl:497-500); it is used
        // the same way here, up to 32 bits: the input triple is checked at 32 random points with b-bit coordinates, exactly over Q
        // (plo_mmchecker_bits) or modulo -m/-q/-r.
        if (a[1] == 'b')
          std::cerr << "# \033[1;33mNOTE: -b " << flags.bitsize << ": 32 random points with " << (flags.bitsize > 32 ? 32 : flags.bitsize) << "-bit coordinates (at most 32 bits here)\033[0m" << std::endl;
      }
      else if (a[1] == 'O' && i + 1 < argc) loops = strtoull(argv[++i], nullptr, 10);
      else if (a[1] == 's') measure = PLO_MEASURE_NNZ;
      else if (a[1] == 'g') measure = PLO_MEASURE_G2;
      else { std::cerr << "# \033[1;31m****** ERROR, option " << a << " is out of scope of this engine ******\033[0m" << std::endl; return -1; }
    } else files.push_back(a);
  }
  if (const int rc = flags.conflict()) return rc;
  if (files.size() < 3) usage(argv[0], loops);
  cli::Triple T(flags.quad, flags.d);
  if (!T.read(files)) return -1;
  // The reference only warns here (its `return 2` is commented out, src/orbiter.cpp:236-242) and then fails inside LinBox; this
  // engine takes flat r x cols buffers, so a mismatched triple is rejected with fMMchecker's code (src/MMchecker.cpp:65-71).
  if (!T.inner_ok()) return T.inner_mismatch();
  uint32_t cnt[2];
  const int v0 = T.check(flags.modulus, flags.bits(), seed, 32, cnt, nullptr);  // :251 (result ignored by the reference)
  int m, k, n;
  plo_LRP2MM(T.cols(0), T.cols(1), T.rows(2), &m, &k, &n);
  verdict_line(v0, m, k, n, cnt[0], cnt[1]);
  if (flags.modulus > 0 && measure != PLO_MEASURE_NNZ) { std::cerr << "# \033[1;31m****** ERROR, -g needs the rationals ******\033[0m" << std::endl; return -1; }
  plo_orbiter_report rep;
  cli::Triple out;
  cli::Timer timer;
  const int rc = T.orbiter(flags.modulus, measure, mode, seed, loops, out, &rep);
  if (rc != PLO_OK) { std::cerr << "# \033[1;31m****** ERROR " << rc << ": " << plo_last_error() << " ******\033[0m" << std::endl; return rc; }
  std::clog << "# Init. ops: " << rep.init_score << ", {" << rep.init_nnz << ',' << rep.init_nno << '}' << std::endl;
  if (flags.modulus == 0 && rep.improved) {
    std::vector<plo_orbit_best> recs(256);
    uint64_t nrec = 0;
    if (T.progress(measure, mode, seed, loops, recs, &nrec) == PLO_OK) found_lines(rep, recs, nrec);
  }
  std::clog << "# Search(" << loops << "): " << timer.seconds() << "s" << std::endl;
  if (rep.improved) {
    reduced_line(rep);
    out.write_nnz(files);
    verdict_line(rep.mm_verdict, m, k, n, rep.best.nnz, rep.best.nno);
  }
  return 0;
}
