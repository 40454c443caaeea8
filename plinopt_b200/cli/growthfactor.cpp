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
  cli::Triple T(quad, d);
  if (!T.read(files)) return -1;
  if (!T.inner_ok()) return T.inner_mismatch();  // :163-169
  int m, k, n;
  plo_LRP2MM(T.cols(0), T.cols(1), T.rows(2), &m, &k, &n);
  double g[11];
  const int rc = T.growth_factors(g);
  if (rc != PLO_OK) { std::cerr << "# \033[1;31m****** ERROR " << rc << ": " << plo_last_error() << " ******\033[0m" << std::endl; return rc; }
  std::clog << "# Norms of " << m << 'x' << k << 'x' << n << " Matrix-Multiplication:" << std::endl;
  const char* names[11] = {"## Ginfinf:\t", "## Ginf2:\t", "## G2inf:\t", "## G22:\t\t", "## G2:\t\t", "## Q0:\t\t", "## Qkinfinf:\t", "## Q1inf2:\t",
                           "## Qk12inf:\t", "## Qk2inf:\t", "## Q122:\t"};
  std::clog << std::fixed << std::setw(8) << "#  \t\tGamma \t\tlog_" << k << std::endl;
  for (int t = 0; t < 11; ++t) std::clog << names[t] << g[t] << '\t' << std::log(g[t]) / std::log((double)k) << std::endl;
  return 0;
}
