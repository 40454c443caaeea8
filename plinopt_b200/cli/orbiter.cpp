// bin/orbiter -- drop-in for src/orbiter.cpp:365-441: random DeGroote-orbit search writing
// <stem>.nnz.sms next to every input when the winner improves on it (:338-348).
// Flags of the reference are kept; -P "X^2-d" searches over Q(sqrt d) (entries a + bX), while -z/-c
// (SLP-operation and canonical measures), -I and other polynomials are out of scope and rejected.
// Added: -g (minimise the growth factor G2 instead of the sparsity), --seed N, --exhaustive, --any-shape.
#include <algorithm>
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

// orbiter -P "X^2-d": the same run over Q(sqrt d), files in X syntax
static int run_quad(int64_t d, const std::vector<std::string>& files, int bits, int measure, int mode, uint64_t seed, uint64_t loops) {
  cli::QuadTriple T;
  if (!T.read(files)) return -1;
  if (T.A[0].rows != T.A[1].rows || T.A[0].rows != T.A[2].cols) {
    std::cerr << "# \033[1;31m****** ERROR, inner dimension mismatch: " << T.A[0].rows << "(.)" << T.A[1].rows << '|' << T.A[2].cols << " ******\033[0m" << std::endl;
    return 2;
  }
  std::vector<cli::NumDen> in;  // La, Lb, Ra, Rb, Pa, Pb
  for (int t = 0; t < 3; ++t) { in.push_back(cli::flatten(T.A[t])); in.push_back(cli::flatten(T.B[t])); }
  const int r = in[0].rows, Lcols = in[0].cols, Rcols = in[2].cols, Prows = in[4].rows;
  const int64_t* q[12];
  for (int x = 0; x < 6; ++x) { q[2 * x] = in[(size_t)x].num.data(); q[2 * x + 1] = in[(size_t)x].den.data(); }
  uint32_t cnt[2];
  const int v0 = plo_mmchecker_quad(d, bits, seed, 32, r, Lcols, in[2].rows, Rcols, Prows, in[4].cols, q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9],
                                    q[10], q[11], cnt, nullptr);
  int m, k, n;
  plo_LRP2MM(Lcols, Rcols, Prows, &m, &k, &n);
  verdict_line(v0, m, k, n, cnt[0], cnt[1]);
  std::vector<std::vector<int64_t>> out(12);
  int64_t* o[12];
  for (int x = 0; x < 12; ++x) { out[(size_t)x].resize(in[(size_t)x / 2].num.size()); o[x] = out[(size_t)x].data(); }
  plo_orbiter_report rep;
  cli::Timer timer;
  const int rc = plo_orbiter_quad(d, measure, mode, seed, loops, r, Lcols, Rcols, Prows, q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9], q[10], q[11],
                                  o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7], o[8], o[9], o[10], o[11], &rep);
  if (rc != PLO_OK) { std::cerr << "# \033[1;31m****** ERROR " << rc << ": " << plo_last_error() << " ******\033[0m" << std::endl; return rc; }
  std::clog << "# Init. ops: " << rep.init_score << ", {" << rep.init_nnz << ',' << rep.init_nno << '}' << std::endl;
  if (rep.improved) {
    std::vector<plo_orbit_best> recs(256);
    uint64_t nrec = 0;
    if (plo_orbiter_progress_quad(d, measure, mode, seed, loops, r, Lcols, Rcols, Prows, q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9], q[10], q[11],
                                  recs.size(), recs.data(), &nrec) == PLO_OK)
      found_lines(rep, recs, nrec);
  }
  std::clog << "# Search(" << loops << "): " << timer.seconds() << "s" << std::endl;
  if (rep.improved) {
    reduced_line(rep);
    for (int t = 0; t < 3; ++t) {
      const cli::NumDen& a = in[2 * (size_t)t];
      std::ofstream f(cli::replace_extension(files[(size_t)t], ".nnz.sms"));
      plo::host::write_sms_quad(f, cli::unflatten(a.rows, a.cols, out[4 * (size_t)t], out[4 * (size_t)t + 1]),
                                cli::unflatten(a.rows, a.cols, out[4 * (size_t)t + 2], out[4 * (size_t)t + 3]));
    }
    verdict_line(rep.mm_verdict, m, k, n, rep.best.nnz, rep.best.nno);
  }
  return 0;
}

int main(int argc, char** argv) {
  unsigned long long loops = 100, modulus = 0, seed = 0x504C494E4F505431ull, bitsize = 32;  // DEFAULT_RANDOM_LOOPS, plinopt_library.h:37-39
  int measure = PLO_MEASURE_NNZ, mode = PLO_MODE_PHILOX;
  bool modular = false, quad = false;
  int64_t d = 0;
  std::vector<std::string> files;
  for (int i = 1; i < argc; ++i) {
    const std::string a(argv[i]);
    if (a == "--seed" && i + 1 < argc) seed = strtoull(argv[++i], nullptr, 0);
    else if (a == "--gpus" && i + 1 < argc) plo_set_sweep_devices(atoi(argv[++i]));
    else if (a == "--exhaustive") mode = PLO_MODE_EXHAUSTIVE;
    else if (a == "--any-shape") plo_set_orbit_any_shape(1);
    else if (a[0] == '-' && a.size() > 1) {
      if (a[1] == 'h') usage(argv[0], loops);
      else if (a[1] == 'b' && i + 1 < argc) {
        // -b is the bit size of the random integer inputs of the reference's over-Q check (plinopt_library.inl:497-500); it is used
        // the same way here, up to 32 bits: the input triple is checked at 32 random points with b-bit coordinates, exactly over Q
        // (plo_mmchecker_bits) or modulo -m/-q/-r.
        bitsize = strtoull(argv[++i], nullptr, 10);
        std::cerr << "# \033[1;33mNOTE: -b " << bitsize << ": 32 random points with " << (bitsize > 32 ? 32 : bitsize) << "-bit coordinates (at most 32 bits here)\033[0m" << std::endl;
      }
      else if ((a[1] == 'm' || a[1] == 'q') && i + 1 < argc) { modulus = strtoull(argv[++i], nullptr, 10); modular = true; }
      else if (a[1] == 'r' && i + 3 < argc) {
        const unsigned long long r = strtoull(argv[++i], nullptr, 10); const int e = atoi(argv[++i]); const unsigned long long s = strtoull(argv[++i], nullptr, 10);
        unsigned long long pw = 1; for (int t = 0; t < e; ++t) pw *= r;
        modulus = pw - s;
        modular = true;
      } else if (a[1] == 'P' && i + 1 < argc) {
        if (!cli::parse_quadratic_modulus(argv[++i], d)) return cli::refuse(std::string("-P \"") + argv[i] + "\": only X^2-d, d an integer, is supported");
        quad = true;
      } else if (a[1] == 'I') return cli::refuse("-I is out of scope of this engine (of the polynomial modes, only -P \"X^2-d\" is supported)");
      else if (a[1] == 'O' && i + 1 < argc) loops = strtoull(argv[++i], nullptr, 10);
      else if (a[1] == 's') measure = PLO_MEASURE_NNZ;
      else if (a[1] == 'g') measure = PLO_MEASURE_G2;
      else { std::cerr << "# \033[1;31m****** ERROR, option " << a << " is out of scope of this engine ******\033[0m" << std::endl; return -1; }
    } else files.push_back(a);
  }
  if (quad && modular) return cli::refuse("-P cannot be combined with -m/-q/-r");
  if (files.size() < 3) usage(argv[0], loops);
  if (quad) return run_quad(d, files, (int)(bitsize < 1 ? 1 : (bitsize > 32 ? 32 : bitsize)), measure, mode, seed, loops);
  plo::host::QField Q;
  plo::host::Dense<plo::host::QField> L, R, P;
  if (!cli::read_file(files[0], L) || !cli::read_file(files[1], R) || !cli::read_file(files[2], P)) return -1;
  if (L.rows != R.rows || L.rows != P.cols) {
    // The reference only warns here (its `return 2` is commented out, src/orbiter.cpp:236-242) and then fails inside LinBox; this
    // engine takes flat r x cols buffers, so a mismatched triple is rejected with fMMchecker's code (src/MMchecker.cpp:65-71).
    std::cerr << "# \033[1;31m****** ERROR, inner dimension mismatch: " << L.rows << "(.)" << R.rows << '|' << P.cols << " ******\033[0m" << std::endl;
    return 2;
  }
  const cli::NumDen l = cli::flatten(L), r = cli::flatten(R), p = cli::flatten(P);
  uint32_t cnt[2];
  const int v0 = plo_mmchecker_bits(modulus, (int)(bitsize < 1 ? 1 : (bitsize > 32 ? 32 : bitsize)), seed, 32, l.rows, l.cols, r.rows, r.cols, p.rows, p.cols, l.num.data(), l.den.data(),
                                    r.num.data(), r.den.data(), p.num.data(), p.den.data(), cnt, nullptr);  // :251 (result ignored by the reference)
  int m, k, n;
  plo_LRP2MM(l.cols, r.cols, p.rows, &m, &k, &n);
  verdict_line(v0, m, k, n, cnt[0], cnt[1]);
  std::vector<int64_t> oLn(l.num.size()), oLd(l.num.size()), oRn(r.num.size()), oRd(r.num.size()), oPn(p.num.size()), oPd(p.num.size());
  plo_orbiter_report rep;
  cli::Timer timer;
  int rc;
  if (modulus > 0) {  // Orbiter<0>()(QQ, F, ...): the search runs in Z/pZ (src/orbiter.cpp:419-426)
    if (measure != PLO_MEASURE_NNZ) { std::cerr << "# \033[1;31m****** ERROR, -g needs the rationals ******\033[0m" << std::endl; return -1; }
    std::fill(oLd.begin(), oLd.end(), 1); std::fill(oRd.begin(), oRd.end(), 1); std::fill(oPd.begin(), oPd.end(), 1);
    rc = plo_orbiter_modp(modulus, mode, seed, loops, l.rows, l.cols, r.cols, p.rows, l.num.data(), l.den.data(), r.num.data(), r.den.data(), p.num.data(),
                          p.den.data(), oLn.data(), oRn.data(), oPn.data(), &rep);
  } else
    rc = plo_orbiter(measure, mode, seed, loops, l.rows, l.cols, r.cols, p.rows, l.num.data(), l.den.data(), r.num.data(), r.den.data(), p.num.data(),
                     p.den.data(), oLn.data(), oLd.data(), oRn.data(), oRd.data(), oPn.data(), oPd.data(), &rep);
  if (rc != PLO_OK) { std::cerr << "# \033[1;31m****** ERROR " << rc << ": " << plo_last_error() << " ******\033[0m" << std::endl; return rc; }
  std::clog << "# Init. ops: " << rep.init_score << ", {" << rep.init_nnz << ',' << rep.init_nno << '}' << std::endl;
  if (modulus == 0 && rep.improved) {
    std::vector<plo_orbit_best> recs(256);
    uint64_t nrec = 0;
    if (plo_orbiter_progress(measure, mode, seed, loops, l.rows, l.cols, r.cols, p.rows, l.num.data(), l.den.data(), r.num.data(), r.den.data(), p.num.data(),
                             p.den.data(), recs.size(), recs.data(), &nrec) == PLO_OK)
      found_lines(rep, recs, nrec);
  }
  std::clog << "# Search(" << loops << "): " << timer.seconds() << "s" << std::endl;
  if (rep.improved) {
    reduced_line(rep);
    const auto Lj = cli::unflatten(l.rows, l.cols, oLn, oLd), Rg = cli::unflatten(r.rows, r.cols, oRn, oRd), hP = cli::unflatten(p.rows, p.cols, oPn, oPd);
    std::ofstream ol(cli::replace_extension(files[0], ".nnz.sms")), orr(cli::replace_extension(files[1], ".nnz.sms")), op(cli::replace_extension(files[2], ".nnz.sms"));
    plo::host::write_matrix(ol, Q, Lj, plo::host::FF_SMS);
    plo::host::write_matrix(orr, Q, Rg, plo::host::FF_SMS);
    plo::host::write_matrix(op, Q, hP, plo::host::FF_SMS);
    verdict_line(rep.mm_verdict, m, k, n, rep.best.nnz, rep.best.nno);
  }
  return 0;
}
