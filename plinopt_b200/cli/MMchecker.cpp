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
  unsigned long long bitsize = 32, modulus = 0, seed = 0x504C494E4F505431ull, samples = 32;
  bool modular = false, quad = false;
  int64_t d = 0;
  std::vector<std::string> files;
  for (int i = 1; i < argc; ++i) {
    const std::string a(argv[i]);
    if (a == "--seed" && i + 1 < argc) seed = strtoull(argv[++i], nullptr, 0);
    else if (a == "--samples" && i + 1 < argc) samples = strtoull(argv[++i], nullptr, 10);
    else if (a[0] == '-' && a.size() > 1) {
      if (a[1] == 'h') usage(argv[0]);
      else if (a[1] == 'b' && i + 1 < argc) bitsize = strtoull(argv[++i], nullptr, 10);
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
      else { std::cerr << "# \033[1;31m****** ERROR, option " << a << " is out of scope of this engine ******\033[0m" << std::endl; return -1; }
    } else files.push_back(a);
  }
  if (quad && modular) return cli::refuse("-P cannot be combined with -m/-q/-r");
  if (files.size() < 3) usage(argv[0]);
  uint32_t cnt[2] = {0, 0};
  const int batch = (int)(samples < 1 ? 1 : (samples > 4096 ? 4096 : samples));
  const int bits = (int)(bitsize < 1 ? 1 : (bitsize > 32 ? 32 : bitsize));
  int nprimes = 0, v;
  cli::NumDen l, r, p;
  if (quad) {
    cli::QuadTriple T;
    if (!T.read(files)) return -1;
    l = cli::flatten(T.A[0]); r = cli::flatten(T.A[1]); p = cli::flatten(T.A[2]);
    const cli::NumDen lb = cli::flatten(T.B[0]), rb = cli::flatten(T.B[1]), pb = cli::flatten(T.B[2]);
    if (bitsize > 32) std::clog << "# NOTE: -b " << bitsize << ": coordinates of at most 32 bits are drawn here (over Q(sqrt d) the verdict is exact at every sampled point either way)" << std::endl;
    v = plo_mmchecker_quad(d, bits, seed, batch, l.rows, l.cols, r.rows, r.cols, p.rows, p.cols, l.num.data(), l.den.data(), lb.num.data(), lb.den.data(),
                           r.num.data(), r.den.data(), rb.num.data(), rb.den.data(), p.num.data(), p.den.data(), pb.num.data(), pb.den.data(), cnt, &nprimes);
    if (v >= 0 && v <= 1) std::clog << "# over Q(sqrt " << d << "): " << batch << " points of " << bits << "-bit coordinates, decided modulo " << nprimes << " word-size prime(s), two embeddings each" << std::endl;
  } else {
    plo::host::Dense<plo::host::QField> L, R, P;
    if (!cli::read_file(files[0], L) || !cli::read_file(files[1], R) || !cli::read_file(files[2], P)) return -1;
    l = cli::flatten(L); r = cli::flatten(R); p = cli::flatten(P);
    if (bitsize > 32) std::clog << "# NOTE: -b " << bitsize << ": coordinates of at most 32 bits are drawn here (over Q the verdict is exact at every sampled point either way)" << std::endl;
    v = plo_mmchecker_bits(modulus, bits, seed, batch, l.rows, l.cols, r.rows, r.cols, p.rows, p.cols,
                           l.num.data(), l.den.data(), r.num.data(), r.den.data(), p.num.data(), p.den.data(), cnt, &nprimes);
    if (modulus == 0 && v >= 0 && v <= 1) std::clog << "# over Q: " << batch << " points of " << (bitsize > 32 ? 32 : bitsize) << "-bit coordinates, decided modulo " << nprimes << " word-size prime(s)" << std::endl;
  }
  int m, k, n;
  plo_LRP2MM(l.cols, r.cols, p.rows, &m, &k, &n);
  if (v == 2) std::cerr << "# \033[1;31m****** ERROR, inner dimension mismatch: " << l.rows << "(.)" << r.rows << '|' << p.cols << " ******\033[0m" << std::endl;
  else if (v == 3) std::cerr << "# \033[1;31m****** ERROR, outer dimension mismatch: " << l.cols << ':' << m << 'x' << k << ' ' << r.cols << ':' << k << 'x' << n << ' ' << p.rows << ':' << m << 'x' << n << " ******\033[0m" << std::endl;
  else if (v == 0) std::clog << "# \033[1;32mSUCCESS: correct " << m << 'x' << k << 'x' << n << " {" << cnt[0] << ',' << cnt[1] << "} Matrix-Multiplication \033[0m" << std::endl;
  else if (v == 1) std::cerr << "# \033[1;31m****** ERROR, not a " << m << 'x' << k << 'x' << n << " MM algorithm******\033[0m" << std::endl;
  else std::cerr << "# \033[1;31m****** ERROR " << v << ": " << plo_last_error() << " ******\033[0m" << std::endl;
  return v;
}
