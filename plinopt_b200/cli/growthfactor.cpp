// bin/growthfactor -- drop-in for src/growthfactor.cpp:148-231: the growth / error factors of an <m x k x n> algorithm,
// printed in the reference's format ("## G2:\t\t<gamma>\t<log_k gamma>").  -P "X^2-d": entries a + bX in Q(sqrt d), d > 0.
#include <cmath>
#include <cstdlib>
#include <iomanip>

#include "cli_common.hpp"

int main(int argc, char** argv) {
  bool quad = false, modular = false;
  int64_t d = 0;
  std::vector<std::string> files;
  for (int i = 1; i < argc; ++i) {
    const std::string a(argv[i]);
    if (a == "-P" && i + 1 < argc) {
      if (!cli::parse_quadratic_modulus(argv[++i], d)) return cli::refuse(std::string("-P \"") + argv[i] + "\": only X^2-d, d an integer, is supported");
      quad = true;
    } else if (a == "-I") return cli::refuse("-I is out of scope of this engine (of the polynomial modes, only -P \"X^2-d\" is supported)");
    else {
      modular = modular || a == "-m" || a == "-q" || a == "-r";  // options of MMchecker and orbiter; without -P read as file names, as before
      files.push_back(a);
    }
  }
  if (quad && modular) return cli::refuse("-P cannot be combined with -m/-q/-r");
  if (files.size() < 3 || files[0] == "-h") { std::clog << "Usage:" << argv[0] << " [-P \"X^2-d\"] L.sms R.sms P.sms\n"; exit(-1); }
  cli::QuadTriple T;  // without -P, the parts in X stay empty
  if (!(quad ? T.read(files) : cli::read_file(files[0], T.A[0]) && cli::read_file(files[1], T.A[1]) && cli::read_file(files[2], T.A[2]))) return -1;
  const plo::host::Dense<plo::host::QField>&L = T.A[0], &R = T.A[1], &P = T.A[2];
  if (L.rows != R.rows || L.rows != P.cols) {  // :163-169
    std::cerr << "# \033[1;31m****** ERROR, inner dimension mismatch: " << L.rows << "(.)" << R.rows << '|' << P.cols << " ******\033[0m" << std::endl;
    return 2;
  }
  const cli::NumDen l = cli::flatten(L), r = cli::flatten(R), p = cli::flatten(P);
  int m, k, n;
  plo_LRP2MM(l.cols, r.cols, p.rows, &m, &k, &n);
  double g[11];
  int rc;
  if (quad) {
    const cli::NumDen lb = cli::flatten(T.B[0]), rb = cli::flatten(T.B[1]), pb = cli::flatten(T.B[2]);
    rc = plo_growth_factors_quad(d, l.rows, l.cols, r.cols, p.rows, l.num.data(), l.den.data(), lb.num.data(), lb.den.data(), r.num.data(), r.den.data(),
                                 rb.num.data(), rb.den.data(), p.num.data(), p.den.data(), pb.num.data(), pb.den.data(), g);
  } else {
    rc = plo_growth_factors(l.rows, l.cols, r.cols, p.rows, l.num.data(), l.den.data(), r.num.data(), r.den.data(), p.num.data(), p.den.data(), g);
  }
  if (rc != PLO_OK) { std::cerr << "# \033[1;31m****** ERROR " << rc << ": " << plo_last_error() << " ******\033[0m" << std::endl; return rc; }
  std::clog << "# Norms of " << m << 'x' << k << 'x' << n << " Matrix-Multiplication:" << std::endl;
  const char* names[11] = {"## Ginfinf:\t", "## Ginf2:\t", "## G2inf:\t", "## G22:\t\t", "## G2:\t\t", "## Q0:\t\t", "## Qkinfinf:\t", "## Q1inf2:\t",
                           "## Qk12inf:\t", "## Qk2inf:\t", "## Q122:\t"};
  std::clog << std::fixed << std::setw(8) << "#  \t\tGamma \t\tlog_" << k << std::endl;
  for (int t = 0; t < 11; ++t) std::clog << names[t] << g[t] << '\t' << std::log(g[t]) / std::log((double)k) << std::endl;
  return 0;
}
