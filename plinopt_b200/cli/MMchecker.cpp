// bin/MMchecker -- drop-in for src/MMchecker.cpp:85-138: Q, mod-m and, of the polynomial modes, -P "X^2-d" (entries a + bX in
// Q(sqrt d)); -I and other polynomials are out of scope.
#include <cstdlib>

#include "cli_common.hpp"

static void usage(const char* prg) {
  std::clog << "Usage: " << prg << " [-h|-b #|-m/-q #|-r # # #|-P \"X^2-d\"|--samples #] L.sms R.sms P.sms\n"
            << "  [-b b]: random check with values of size 'bitsize' (default 32; at most 32 here)\n"
            << "  [--samples s]: number of random points checked (default 32; the reference checks one)\n"
            << "  [-m/-q m]: check is modulo (mod) or (mod/2^k) (default no)\n"
            << "  [-r r e s]: check is modulo (r^e-s) or ((r^e-s)/2^k) (default no)\n"
            << "  [-P \"X^2-d\"]: entries a+bX in Q(sqrt d), X^2 = d (default no)\n";
  exit(-1);
}

int main(int argc, char** argv) {
  unsigned long long seed = 0x504C494E4F505431ull, samples = 32;
  cli::CheckFlags flags;
  std::vector<std::string> files;
  for (int i = 1; i < argc; ++i) {
    const std::string a(argv[i]);
    if (a == "--seed" && i + 1 < argc) seed = strtoull(argv[++i], nullptr, 0);
    else if (a == "--samples" && i + 1 < argc) samples = strtoull(argv[++i], nullptr, 10);
    else if (a[0] == '-' && a.size() > 1) {
      if (a[1] == 'h') usage(argv[0]);
      else if (const int t = flags.take(argc, argv, i)) { if (t < 0) return -1; }
      else { std::cerr << "# \033[1;31m****** ERROR, option " << a << " is out of scope of this engine ******\033[0m" << std::endl; return -1; }
    } else files.push_back(a);
  }
  if (const int rc = flags.conflict()) return rc;
  if (files.size() < 3) usage(argv[0]);
  uint32_t cnt[2] = {0, 0};
  const int batch = (int)(samples < 1 ? 1 : (samples > 4096 ? 4096 : samples));
  int nprimes = 0;
  cli::Triple T(flags.quad, flags.d);
  if (!T.read(files)) return -1;
  if (flags.bitsize > 32)
    std::clog << "# NOTE: -b " << flags.bitsize << ": coordinates of at most 32 bits are drawn here (over " << (flags.quad ? "Q(sqrt d)" : "Q") << " the verdict is exact at every sampled point either way)" << std::endl;
  const int v = T.check(flags.modulus, flags.bits(), seed, batch, cnt, &nprimes);
  if (flags.modulus == 0 && v >= 0 && v <= 1)  // over Q the bit size as given, at most 32
    std::clog << "# over " << (flags.quad ? "Q(sqrt " + std::to_string(flags.d) + ")" : "Q") << ": " << batch << " points of " << (flags.quad ? flags.bits() : std::min(flags.bitsize, 32ull))
              << "-bit coordinates, decided modulo " << nprimes << " word-size prime(s)" << (flags.quad ? ", two embeddings each" : "") << std::endl;
  int m, k, n;
  plo_LRP2MM(T.cols(0), T.cols(1), T.rows(2), &m, &k, &n);
  if (v == 2) T.inner_mismatch();
  else if (v == 3) std::cerr << "# \033[1;31m****** ERROR, outer dimension mismatch: " << T.cols(0) << ':' << m << 'x' << k << ' ' << T.cols(1) << ':' << k << 'x' << n << ' ' << T.rows(2) << ':' << m << 'x' << n << " ******\033[0m" << std::endl;
  else if (v == 0) std::clog << "# \033[1;32mSUCCESS: correct " << m << 'x' << k << 'x' << n << " {" << cnt[0] << ',' << cnt[1] << "} Matrix-Multiplication \033[0m" << std::endl;
  else if (v == 1) std::cerr << "# \033[1;31m****** ERROR, not a " << m << 'x' << k << 'x' << n << " MM algorithm******\033[0m" << std::endl;
  else std::cerr << "# \033[1;31m****** ERROR " << v << ": " << plo_last_error() << " ******\033[0m" << std::endl;
  return v;
}
