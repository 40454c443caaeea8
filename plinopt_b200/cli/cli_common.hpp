// cli_common.hpp -- shared pieces of the drop-in CLIs (bin/sparsifier, bin/orbiter, bin/MMchecker, ...).
#pragma once
#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "../../include/plinopt_b200.h"
#include "../csrc/host/matrix_io.hpp"

namespace cli {

using plo::host::Dense;
using plo::host::QField;
using plo::host::Rat;

struct NumDen {
  std::vector<int64_t> num, den;
  int rows = 0, cols = 0;
};

inline NumDen flatten(const Dense<QField>& M) {
  NumDen o;
  o.rows = (int)M.rows; o.cols = (int)M.cols;
  o.num.resize(M.v.size()); o.den.resize(M.v.size());
  for (size_t e = 0; e < M.v.size(); ++e) { o.num[e] = M.v[e].num; o.den[e] = M.v[e].den; }
  return o;
}
inline Dense<QField> unflatten(int rows, int cols, const std::vector<int64_t>& num, const std::vector<int64_t>& den) {
  QField Q;
  Dense<QField> M(Q, (size_t)rows, (size_t)cols);
  for (size_t e = 0; e < M.v.size(); ++e) M.v[e] = Rat::make(num[e], den[e]);
  return M;
}
inline int refuse(const std::string& why) {  // an option outside what this engine does: exit code -1
  std::cerr << "# \033[1;31m****** ERROR, " << why << " ******\033[0m" << std::endl;
  return -1;
}
// SMS file through `read`: read_sms, or read_sms_quad (entries a + bX) under -P
template <class Read>
bool read_file_with(const std::string& name, Read read) {
  std::ifstream in(name);
  if (!in) { std::cerr << "# \033[1;31m****** ERROR, cannot open " << name << " ******\033[0m" << std::endl; return false; }
  try {
    if (!read(in)) { std::cerr << "# \033[1;31m****** ERROR, malformed SMS file " << name << " ******\033[0m" << std::endl; return false; }
  } catch (const std::exception& e) {
    std::cerr << "# \033[1;31m****** ERROR, " << name << ": " << e.what() << " ******\033[0m" << std::endl;
    return false;
  }
  return true;
}
inline bool read_file(const std::string& name, Dense<QField>& M) {
  return read_file_with(name, [&](std::istream& in) { return plo::host::read_sms(in, M); });
}
inline std::string replace_extension(const std::string& path, const std::string& ext) {  // std::filesystem::path::replace_extension
  const size_t slash = path.find_last_of('/');
  const size_t dot = path.find_last_of('.');
  if (dot == std::string::npos || (slash != std::string::npos && dot < slash)) return path + ext;
  return path.substr(0, dot) + ext;
}

// -P of MMchecker, orbiter and growthfactor: the field Q(sqrt d) of the polynomial X^2 - d.  Spaces are ignored; `X^2-d` and `X^2+d`
// with d an integer are accepted, any other polynomial is refused (false).  Whether X^2 - d is irreducible is the library's check.
inline bool parse_quadratic_modulus(const std::string& poly, int64_t& d) {
  std::string t;
  for (char c : poly) if (c != ' ' && c != '\t') t += c;
  if (t.size() < 5 || t.compare(0, 3, "X^2") != 0 || (t[3] != '-' && t[3] != '+')) return false;
  const std::string digits = t.substr(4);
  if (digits.find_first_not_of("0123456789") != std::string::npos || digits.size() > 18) return false;
  const int64_t v = std::stoll(digits);
  d = t[3] == '-' ? v : -v;
  return true;
}
// The flags MMchecker and orbiter share: -b (bit size of the random points), -m/-q and -r r e s (a check modulo m or r^e - s),
// -P "X^2-d" (entries a + bX in Q(sqrt d)); -I is refused.
struct CheckFlags {
  unsigned long long bitsize = 32, modulus = 0;  // bitsize as given
  bool modular = false, quad = false;
  int64_t d = 0;
  int bits() const { return (int)(bitsize < 1 ? 1 : (bitsize > 32 ? 32 : bitsize)); }
  // argv[i] if it is one of these flags, with its arguments (i moves past them): 1, or -1 after a refusal; 0 for any other argument
  int take(int argc, char** argv, int& i) {
    const char f = argv[i][1];
    if (f == 'b' && i + 1 < argc) bitsize = strtoull(argv[++i], nullptr, 10);
    else if ((f == 'm' || f == 'q') && i + 1 < argc) { modulus = strtoull(argv[++i], nullptr, 10); modular = true; }
    else if (f == 'r' && i + 3 < argc) {
      const unsigned long long r = strtoull(argv[++i], nullptr, 10); const int e = atoi(argv[++i]); const unsigned long long s = strtoull(argv[++i], nullptr, 10);
      unsigned long long pw = 1; for (int t = 0; t < e; ++t) pw *= r;
      modulus = pw - s;
      modular = true;
    } else if (f == 'P' && i + 1 < argc) {
      if (!parse_quadratic_modulus(argv[++i], d)) return refuse(std::string("-P \"") + argv[i] + "\": only X^2-d, d an integer, is supported");
      quad = true;
    } else if (f == 'I') return refuse("-I is out of scope of this engine (of the polynomial modes, only -P \"X^2-d\" is supported)");
    else return 0;
    return 1;
  }
  // after the last flag: -1 for -P with -m/-q/-r, else 0
  int conflict() const { return quad && modular ? refuse("-P cannot be combined with -m/-q/-r") : 0; }
};

// A triple read from three SMS files: over Q, A[t] are the matrices and B stays empty; over Q(sqrt d) (-P "X^2-d", entries a + bX),
// A[t] are the rational parts and B[t] the parts in X.  Its calls are the only place that chooses between an entry point over Q and
// its _quad twin.
struct Triple {
  bool quad;
  int64_t d;
  Dense<QField> A[3], B[3];

  explicit Triple(bool quadratic = false, int64_t radicand = 0) : quad(quadratic), d(radicand) {}
  int rows(int t) const { return (int)A[t].rows; }
  int cols(int t) const { return (int)A[t].cols; }
  bool read(const std::vector<std::string>& files) {
    for (int t = 0; t < 3; ++t)
      if (!read_file_with(files[(size_t)t], [&](std::istream& in) { return quad ? plo::host::read_sms_quad(in, A[t], B[t]) : plo::host::read_sms(in, A[t]); }))
        return false;
    return true;
  }
  bool inner_ok() const { return A[0].rows == A[1].rows && A[0].rows == A[2].cols; }
  int inner_mismatch() const {  // src/MMchecker.cpp:65-71
    std::cerr << "# \033[1;31m****** ERROR, inner dimension mismatch: " << A[0].rows << "(.)" << A[1].rows << '|' << A[2].cols << " ******\033[0m" << std::endl;
    return 2;
  }
  // plo_mmchecker_bits or plo_mmchecker_quad
  int check(uint64_t modulus, int bits, uint64_t seed, int batch, uint32_t* cnt, int* nprimes) const {
    const std::vector<NumDen> f = flat();
    const std::vector<const int64_t*> q = pointers(f);
    if (quad)
      return plo_mmchecker_quad(d, bits, seed, batch, rows(0), cols(0), rows(1), cols(1), rows(2), cols(2), q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8],
                                q[9], q[10], q[11], cnt, nprimes);
    return plo_mmchecker_bits(modulus, bits, seed, batch, rows(0), cols(0), rows(1), cols(1), rows(2), cols(2), q[0], q[1], q[2], q[3], q[4], q[5], cnt, nprimes);
  }
  // plo_orbiter or plo_orbiter_quad; over Q with modulus > 0, plo_orbiter_modp (Orbiter<0>()(QQ, F, ...): the search runs in Z/pZ,
  // src/orbiter.cpp:419-426).  `out` takes the returned triple.
  int orbiter(uint64_t modulus, int measure, int mode, uint64_t seed, uint64_t loops, Triple& out, plo_orbiter_report* rep) const {
    const std::vector<NumDen> f = flat();
    const std::vector<const int64_t*> q = pointers(f);
    std::vector<NumDen> o = f;  // the shapes of the input
    std::vector<int64_t*> w;
    for (NumDen& x : o) { w.push_back(x.num.data()); w.push_back(x.den.data()); }
    const int r = rows(0);
    int rc;
    if (quad)
      rc = plo_orbiter_quad(d, measure, mode, seed, loops, r, cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9], q[10], q[11],
                            w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], w[8], w[9], w[10], w[11], rep);
    else if (modulus > 0) {
      for (NumDen& x : o) std::fill(x.den.begin(), x.den.end(), 1);  // it writes the residues only
      rc = plo_orbiter_modp(modulus, mode, seed, loops, r, cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], w[0], w[2], w[4], rep);
    } else
      rc = plo_orbiter(measure, mode, seed, loops, r, cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], w[0], w[1], w[2], w[3], w[4], w[5], rep);
    out.quad = quad; out.d = d;
    for (int t = 0; t < 3; ++t) {
      const NumDen& a = o[quad ? 2 * (size_t)t : (size_t)t];
      out.A[t] = unflatten(a.rows, a.cols, a.num, a.den);
      if (quad) out.B[t] = unflatten(a.rows, a.cols, o[2 * (size_t)t + 1].num, o[2 * (size_t)t + 1].den);
    }
    return rc;
  }
  // plo_orbiter_progress or plo_orbiter_progress_quad: the '# Found opt:' records
  int progress(int measure, int mode, uint64_t seed, uint64_t loops, std::vector<plo_orbit_best>& recs, uint64_t* nrec) const {
    const std::vector<NumDen> f = flat();
    const std::vector<const int64_t*> q = pointers(f);
    if (quad)
      return plo_orbiter_progress_quad(d, measure, mode, seed, loops, rows(0), cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9],
                                       q[10], q[11], recs.size(), recs.data(), nrec);
    return plo_orbiter_progress(measure, mode, seed, loops, rows(0), cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], recs.size(), recs.data(), nrec);
  }
  // plo_growth_factors or plo_growth_factors_quad
  int growth_factors(double* g) const {
    const std::vector<NumDen> f = flat();
    const std::vector<const int64_t*> q = pointers(f);
    if (quad)
      return plo_growth_factors_quad(d, rows(0), cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9], q[10], q[11], g);
    return plo_growth_factors(rows(0), cols(0), cols(1), rows(2), q[0], q[1], q[2], q[3], q[4], q[5], g);
  }
  // <stem>.nnz.sms next to each input file (src/orbiter.cpp:338-348), in X syntax over Q(sqrt d)
  void write_nnz(const std::vector<std::string>& files) const {
    for (int t = 0; t < 3; ++t) {
      std::ofstream f(replace_extension(files[(size_t)t], ".nnz.sms"));
      if (quad) plo::host::write_sms_quad(f, A[t], B[t]);
      else plo::host::write_matrix(f, QField(), A[t], plo::host::FF_SMS);
    }
  }

  // the arrays of the entry points: A[0], A[1], A[2] over Q; A[0], B[0], A[1], B[1], A[2], B[2] over Q(sqrt d)
  std::vector<NumDen> flat() const {
    std::vector<NumDen> f;
    for (int t = 0; t < 3; ++t) { f.push_back(flatten(A[t])); if (quad) f.push_back(flatten(B[t])); }
    return f;
  }
  static std::vector<const int64_t*> pointers(const std::vector<NumDen>& f) {
    std::vector<const int64_t*> q;
    for (const NumDen& x : f) { q.push_back(x.num.data()); q.push_back(x.den.data()); }
    return q;
  }
};
inline size_t profile(std::ostream& out, const Dense<QField>& M) {  // densityProfile, plinopt_sparsify.inl:118-126
  size_t ss = 0;
  for (size_t i = 0; i < M.rows; ++i) {
    size_t s = 0;
    for (size_t j = 0; j < M.cols; ++j) s += M.at(i, j).num != 0;
    ss += s;
    out << s << ' ';
  }
  out << '=' << ss;
  return ss;
}
struct Timer {
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  double seconds() const { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
};

}  // namespace cli
