// matrix_io.hpp -- SMS reader/writer and the other print formats of the CLIs.
// SMS (reference data/README.md:10-17): optional '#' comment lines, header `rows cols R|M`,
// 1-based `i j value` lines (value = integer or a/b, entries in any order), terminator `0 0 0`.  With `-P "X^2-d"` a value may
// also be a + bX (parse_quadratic).
// Writers follow the shapes LinBox produces for FileFormat(5) SMS (15 `M`-typed files in the
// reference's data/ show it: header `r c M`, row-major entries, `0 0 0`), Maple (1) and a
// bracketed row listing for Pretty (8) / Linalg (12); LinBox's writer itself is not in the
// reference tree (parity unpinned for the pretty layouts).
#pragma once
#include <istream>
#include <ostream>
#include <sstream>
#include <string>

#include "exact.hpp"

namespace plo {
namespace host {

enum FileFormat { FF_MAPLE = 1, FF_SMS = 5, FF_PRETTY = 8, FF_LINALG = 12 };

inline Rat parse_rational(const std::string& tok) {
  const size_t slash = tok.find('/');
  try {
    size_t used = 0;
    const long long n = std::stoll(tok.substr(0, slash), &used);
    if (used != (slash == std::string::npos ? tok.size() : slash)) throw std::invalid_argument(tok);
    if (slash == std::string::npos) return Rat((int64_t)n);
    const std::string ds = tok.substr(slash + 1);
    const long long d = std::stoll(ds, &used);
    if (used != ds.size()) throw std::invalid_argument(tok);
    return Rat::make(n, d);
  } catch (const std::exception&) {
    throw RangeError("cannot parse matrix entry '" + tok + "' (entries in X need -P \"X^2-d\")");
  }
}

// An entry a + b.X of Q(sqrt d), X^2 = d: `q`, `qX`, `X`, `-X`, `q+qX` or `q-qX`, q an integer or n/m as above, the coefficient
// of X omitted for +-1 (`1/2X`, `-3X`, `1/2-X`).  The reference's reader of these files (Givaro) and its `*-X_*` data files are
// not available here: this grammar is a restatement, not checked against them.
inline void parse_quadratic(const std::string& tok, Rat& a, Rat& b) {
  auto bad = [&]() { return RangeError("cannot parse matrix entry '" + tok + "' as a + bX"); };
  a = Rat(); b = Rat();
  if (tok.empty() || tok.back() != 'X') {
    try { a = parse_rational(tok); } catch (const RangeError&) { throw bad(); }
    return;
  }
  const std::string body = tok.substr(0, tok.size() - 1);
  if (body.find('X') != std::string::npos) throw bad();
  size_t split = std::string::npos;  // the sign between q and qX: not the leading one, not one of a denominator
  for (size_t t = 1; t < body.size(); ++t)
    if ((body[t] == '+' || body[t] == '-') && body[t - 1] != '/') split = t;
  const std::string coef = split == std::string::npos ? body : body.substr(split);
  try {
    if (split != std::string::npos) a = parse_rational(body.substr(0, split));
    b = coef.empty() || coef == "+" ? Rat(1) : coef == "-" ? Rat(-1) : parse_rational(coef);
  } catch (const RangeError&) {
    throw bad();
  }
}

// The loop of every SMS reader: comment lines, the header (`header(rows, cols)`), then `entry(i, j, token)` with 0-based i, j for
// each entry line up to `0 0 0`.
template <class Header, class Entry>
bool read_sms_lines(std::istream& in, Header header, Entry entry) {
  std::string line;
  long long rows = -1, cols = -1;
  while (std::getline(in, line)) {
    size_t b = line.find_first_not_of(" \t\r");
    if (b == std::string::npos || line[b] == '#' || line[b] == '%') continue;
    std::istringstream ls(line);
    if (rows < 0) {
      long long r, c;
      if (!(ls >> r >> c) || r < 0 || c < 0) return false;
      rows = r; cols = c;
      header((size_t)r, (size_t)c);
      continue;
    }
    long long i, j;
    std::string val;
    if (!(ls >> i >> j >> val)) return false;
    if (i == 0 && j == 0) break;
    if (i < 1 || j < 1 || i > rows || j > cols) return false;
    entry((size_t)i - 1, (size_t)j - 1, val);
  }
  return rows >= 0;
}

inline bool read_sms(std::istream& in, Dense<QField>& M) {
  QField Q;
  return read_sms_lines(in, [&](size_t r, size_t c) { M = Dense<QField>(Q, r, c); },
                        [&](size_t i, size_t j, const std::string& v) { M.at(i, j) = parse_rational(v); });
}

// A matrix over Q(sqrt d) (`-P "X^2-d"`): A holds the rational parts, B the parts in X.
inline bool read_sms_quad(std::istream& in, Dense<QField>& A, Dense<QField>& B) {
  QField Q;
  return read_sms_lines(in, [&](size_t r, size_t c) { A = Dense<QField>(Q, r, c); B = Dense<QField>(Q, r, c); },
                        [&](size_t i, size_t j, const std::string& v) { parse_quadratic(v, A.at(i, j), B.at(i, j)); });
}

inline void print_elt(std::ostream& o, const Rat& r) { o << r.num; if (r.den != 1) o << '/' << r.den; }
inline void print_elt(std::ostream& o, const int64_t& r) { o << r; }

template <class F>
std::ostream& write_matrix(std::ostream& out, const F& f, const Dense<F>& M, int format) {
  if (format == FF_SMS) {
    out << M.rows << ' ' << M.cols << " M\n";
    for (size_t i = 0; i < M.rows; ++i)
      for (size_t j = 0; j < M.cols; ++j)
        if (!f.is_zero(M.at(i, j))) { out << i + 1 << ' ' << j + 1 << ' '; print_elt(out, M.at(i, j)); out << '\n'; }
    return out << "0 0 0\n";
  }
  if (format == FF_MAPLE) {
    out << "Matrix(" << M.rows << ',' << M.cols << ",[";
    for (size_t i = 0; i < M.rows; ++i) {
      out << (i ? ",[" : "[");
      for (size_t j = 0; j < M.cols; ++j) { if (j) out << ','; print_elt(out, M.at(i, j)); }
      out << ']';
    }
    return out << "])";
  }
  for (size_t i = 0; i < M.rows; ++i) {  // Pretty / Linalg
    out << "  [";
    for (size_t j = 0; j < M.cols; ++j) { out << (j ? " " : ""); print_elt(out, M.at(i, j)); }
    out << " ]\n";
  }
  return out;
}

// SMS of a matrix over Q(sqrt d) in the forms parse_quadratic reads: `a`, `bX` (`X`, `-X`), `a+bX` or `a-|b|X`.
inline std::ostream& write_sms_quad(std::ostream& out, const Dense<QField>& A, const Dense<QField>& B) {
  out << A.rows << ' ' << A.cols << " M\n";
  for (size_t i = 0; i < A.rows; ++i)
    for (size_t j = 0; j < A.cols; ++j) {
      const Rat& a = A.at(i, j);
      Rat b = B.at(i, j);
      if (a.num == 0 && b.num == 0) continue;
      out << i + 1 << ' ' << j + 1 << ' ';
      if (a.num != 0) print_elt(out, a);
      if (b.num != 0) {
        if (b.num < 0) { out << '-'; b.num = -b.num; } else if (a.num != 0) out << '+';
        if (!(b.num == 1 && b.den == 1)) print_elt(out, b);
        out << 'X';
      }
      out << '\n';
    }
  return out << "0 0 0\n";
}

}  // namespace host
}  // namespace plo
