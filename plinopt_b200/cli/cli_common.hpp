// cli_common.hpp -- shared pieces of the drop-in CLIs (bin/sparsifier, bin/orbiter, bin/MMchecker, ...).
#pragma once
#include <chrono>
#include <cstdint>
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
// A triple over Q(sqrt d) read from three SMS files with entries a + bX: A[t] the rational parts, B[t] the parts in X
struct QuadTriple {
  Dense<QField> A[3], B[3];
  bool read(const std::vector<std::string>& files) {
    for (int t = 0; t < 3; ++t)
      if (!read_file_with(files[(size_t)t], [&](std::istream& in) { return plo::host::read_sms_quad(in, A[t], B[t]); })) return false;
    return true;
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
inline std::string replace_extension(const std::string& path, const std::string& ext) {  // std::filesystem::path::replace_extension
  const size_t slash = path.find_last_of('/');
  const size_t dot = path.find_last_of('.');
  if (dot == std::string::npos || (slash != std::string::npos && dot < slash)) return path + ext;
  return path.substr(0, dot) + ext;
}

}  // namespace cli
