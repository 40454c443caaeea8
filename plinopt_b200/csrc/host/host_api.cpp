// host_api.cpp -- extern "C" host-level entry points: the reference's drivers restated around
// the GPU kernels (TSparsifier src/sparsifier.cpp:20-55, Orbiter src/orbiter.cpp:215-360,
// fMMchecker src/MMchecker.cpp:48-81).  No CUDA code here; everything heavy goes through the
// kernel-level C ABI (plo_lincomb_search, plo_orbit_*, plo_mmcheck_*).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <ostream>
#include <streambuf>
#include <vector>

#include <unistd.h>

#include "../plo_device.cuh"
#include "dependency_host.hpp"
#include "factor_host.hpp"
#include "matrix_io.hpp"
#include "negate_host.hpp"
#include "slp.hpp"
#include "sparsify_host.hpp"

using namespace plo::host;

namespace {

// minimal ostream over a file descriptor (progress lines of the reference go to std::clog)
class FdBuf : public std::streambuf {
  int fd_;
 protected:
  int overflow(int c) override { if (c != EOF) { char ch = (char)c; if (::write(fd_, &ch, 1) != 1) return EOF; } return c; }
  std::streamsize xsputn(const char* s, std::streamsize n) override { return ::write(fd_, s, (size_t)n); }
 public:
  explicit FdBuf(int fd) : fd_(fd) {}
};

template <class F>
Dense<F> load(const F& f, size_t r, size_t c, const int64_t* num, const int64_t* den) {
  Dense<F> M(f, r, c);
  for (size_t e = 0; e < r * c; ++e) M.v[e] = f.from_ratio(num[e], den ? den[e] : 1);
  return M;
}
void store(const Dense<QField>& M, int64_t* num, int64_t* den) {
  for (size_t e = 0; e < M.v.size(); ++e) { num[e] = M.v[e].num; if (den) den[e] = M.v[e].den; }
}
void store(const Dense<ZpField>& M, int64_t* num, int64_t* den) {
  for (size_t e = 0; e < M.v.size(); ++e) { num[e] = M.v[e]; if (den) den[e] = 1; }
}

// The body of an entry point with its exceptions as return codes and "<who>: <what>" as the error message
template <class F>
int guarded(const char* who, F&& body) {
  try {
    return body();
  } catch (const EngineError& e) {
    plo::set_error("%s: %s", who, e.what());
    return e.code;
  } catch (const RangeError& e) {
    plo::set_error("%s: %s", who, e.what());
    return PLO_E_RANGE;
  }
}
// <m, k, n> of a triple (library.inl:487-495): 0, or 3 when the outer dimensions do not fit one
int mm_shape(const char* who, int Lcols, int Rcols, int Prows, int* m, int* k, int* n) {
  plo_LRP2MM(Lcols, Rcols, Prows, m, k, n);
  if (Lcols == *m * *k && Rcols == *k * *n && Prows == *m * *n) return 0;
  plo::set_error("%s: outer dimension mismatch", who);
  return 3;
}

template <class F>
int run_sparsifier(const F& f, int rows, int cols, const int64_t* num, const int64_t* den, int blocksize, int maxnumcoeff,
                   int initialElimination, int64_t* cob_num, int64_t* cob_den, int64_t* res_num, int64_t* res_den,
                   int* consistent, uint64_t* stats, std::ostream* log) {
  Dense<F> M = load(f, (size_t)rows, (size_t)cols, num, den);
  Sparsifier<F> sp(f, log);
  if (log) { size_t sc; sp.densityProfile(*log << "# [SPRF] Initial profile: ", sc, M) << std::endl; *log << std::string(30, '#') << std::endl; }
  Dense<F> CoB(f, (size_t)cols, (size_t)cols), Res(f, (size_t)rows, (size_t)cols);
  sp.blockSparsifier(CoB, Res, M, (size_t)blocksize, (size_t)maxnumcoeff, initialElimination != 0);
  store(CoB, cob_num, cob_den);
  store(Res, res_num, res_den);
  if (consistent) *consistent = sp.consistency(M, Res, CoB) ? 1 : 0;
  if (stats) { stats[0] = sp.stats.candidates; stats[1] = sp.stats.searches; stats[2] = sp.stats.fallbacks; }
  if (getenv("PLO_TIMING")) fprintf(stderr, "# [B200] plo_sparsifier: %.1f us inside %llu device round trips; host: begin_alternate %.1f us (incl. first begin_local), begin_local %.1f us, finish_local %.1f us (incl. nested begin_local)\n", sp.stats.device_seconds * 1e6, sp.stats.searches, sp.stats.t_begin_alt * 1e6, sp.stats.t_begin_local * 1e6, sp.stats.t_finish_local * 1e6);
  return PLO_OK;
}

int64_t lcd_of(const int64_t* den, size_t cnt, wide limit = (wide)INT32_MAX) {
  int64_t l = 1;
  for (size_t e = 0; e < cnt; ++e) {
    const int64_t d = den ? (den[e] < 0 ? -den[e] : den[e]) : 1;
    if (d == 0) throw RangeError("zero denominator");
    const wide v = (wide)l / wgcd(l, d) * d;
    if (v > limit) throw RangeError("common denominator too large");
    l = (int64_t)v;
  }
  return l;
}
// scaled to 64-bit integers; `fits32` reports whether every entry (and the common denominator) also fits the int32 C ABI
std::vector<int64_t> scale_int64(const int64_t* num, const int64_t* den, size_t cnt, int64_t lcd, bool& fits32) {
  std::vector<int64_t> out(cnt);
  if (lcd > (int64_t)INT32_MAX) fits32 = false;
  for (size_t e = 0; e < cnt; ++e) {
    const int64_t d = den ? den[e] : 1;
    const wide v = (wide)num[e] * (lcd / d);
    if (wabs(v) >= ((wide)1 << 46)) throw RangeError("scaled entry exceeds 46 bits");
    if (wabs(v) > (wide)INT32_MAX) fits32 = false;
    out[e] = (int64_t)v;
  }
  return out;
}

// plinopt_library.inl:258-269.  Over Q(sqrt d) (B: the sqrt(d) part of M) an entry is zero iff both parts are, and +-1 iff its
// sqrt(d) part is zero and its rational part is +-1 (DESIGN.md 5.1).
void count_nonzeroes(const Dense<QField>& M, uint32_t& nnz, uint32_t& nno, const Dense<QField>* B = nullptr) {
  for (size_t t = 0; t < M.v.size(); ++t) {
    const Rat& e = M.v[t];
    const bool surd = B && B->v[t].num != 0;
    if (e.num != 0 || surd) { ++nnz; if (surd || !(e.den == 1 && (e.num == 1 || e.num == -1))) ++nno; }
  }
}
// growthfactor.cpp:117-125; over Q(sqrt d) (B: the sqrt(d) parts of L, R, P, s = sqrt(d) > 0) every entry a + b.s is a double first
double growth_G2(const Dense<QField>& L, const Dense<QField>& R, const Dense<QField>& P, const Dense<QField>* B = nullptr, double s = 0.) {
  auto x = [&](const Dense<QField>& M, int t, size_t i, size_t j) {
    const double a = (double)M.at(i, j).num / (double)M.at(i, j).den;
    return B ? a + (double)B[t].at(i, j).num / (double)B[t].at(i, j).den * s : a;
  };
  double g = 0.;
  for (size_t i = 0; i < P.cols; ++i) {
    double a = 0., b = 0., c = 0.;
    for (size_t j = 0; j < L.cols; ++j) { const double v = x(L, 0, i, j); a += v * v; }
    for (size_t j = 0; j < R.cols; ++j) { const double v = x(R, 1, i, j); b += v * v; }
    for (size_t j = 0; j < P.rows; ++j) { const double v = x(P, 2, j, i); c += v * v; }
    g += std::sqrt(a) * std::sqrt(b) * std::sqrt(c);
  }
  return g;
}

struct CsrHost {
  std::vector<int64_t> ptr;
  std::vector<int32_t> col;
  std::vector<uint32_t> val;
  plo_csr view(int rows, int cols) const { plo_csr c; c.rows = rows; c.cols = cols; c.ptr = ptr.data(); c.col = col.data(); c.val = val.data(); return c; }
};
// The non-zero entries of a dense rational matrix, row by row (built once; the check over Q reduces them modulo several primes).
// Over Q(sqrt d), B is the sqrt(d) part of the matrix: an entry a + b.sqrt(d) is kept when a or b is non-zero.
struct SparseQ {
  size_t rows = 0, cols = 0;
  std::vector<int64_t> ptr, num, den, bnum, bden;  // bnum, bden: over Q(sqrt d) only
  std::vector<int32_t> col;
  explicit SparseQ(const Dense<QField>& M, const Dense<QField>* B = nullptr) : rows(M.rows), cols(M.cols) {
    ptr.assign(1, 0);
    for (size_t i = 0; i < M.rows; ++i) {
      for (size_t j = 0; j < M.cols; ++j) {
        const Rat& e = M.at(i, j);
        if (e.num == 0 && !(B && B->at(i, j).num != 0)) continue;
        col.push_back((int32_t)j); num.push_back(e.num); den.push_back(e.den);
        if (B) { bnum.push_back(B->at(i, j).num); bden.push_back(B->at(i, j).den); }
      }
      ptr.push_back((int64_t)col.size());
    }
  }
};
// a/b -> a.b^-1 mod p, and over Q(sqrt d) a + b.sqrt(d) -> a + b.root mod p (root^2 = d mod p); returns false if some denominator
// vanishes mod p
bool to_csr(const SparseQ& M, int64_t p, CsrHost& out, int64_t root = 0) {
  ZpField Z(p);
  out.ptr.assign(1, 0); out.col.clear(); out.val.clear();
  int64_t last_den = 1, last_inv = 1;  // few distinct denominators: the last inverse is usually the one needed
  int64_t last_bden = 1, last_binv = 1;
  auto inverse = [&Z](int64_t d, int64_t& last, int64_t& inv) {
    if (d == last) return true;
    if (Z.canon(d) == 0) return false;
    last = d; inv = Z.div(1, Z.canon(d));
    return true;
  };
  for (size_t i = 0; i < M.rows; ++i) {
    for (int64_t t = M.ptr[i]; t < M.ptr[i + 1]; ++t) {
      if (!inverse(M.den[(size_t)t], last_den, last_inv)) return false;
      int64_t v = Z.mul(Z.canon(M.num[(size_t)t]), last_inv);
      if (!M.bnum.empty()) {
        if (!inverse(M.bden[(size_t)t], last_bden, last_binv)) return false;
        v = Z.add(v, Z.mul(Z.mul(Z.canon(M.bnum[(size_t)t]), last_binv), root));
      }
      if (v) { out.col.push_back(M.col[(size_t)t]); out.val.push_back((uint32_t)v); }
    }
    out.ptr.push_back((int64_t)out.col.size());
  }
  return true;
}
// the non-zero entries of a matrix of residues, row by row
void to_csr(const Dense<ZpField>& M, CsrHost& out) {
  out.ptr.assign(1, 0); out.col.clear(); out.val.clear();
  for (size_t i = 0; i < M.rows; ++i) {
    for (size_t j = 0; j < M.cols; ++j) if (M.at(i, j) != 0) { out.col.push_back((int32_t)j); out.val.push_back((uint32_t)M.at(i, j)); }
    out.ptr.push_back((int64_t)out.col.size());
  }
}
bool is_prime(uint64_t x) {
  if (x < 2) return false;
  for (uint64_t d = 2; d * d <= x; ++d) if (x % d == 0) return false;
  return true;
}

// log2 of a common multiple of the denominators of M (the product of the distinct ones, over both parts over Q(sqrt d)) and its
// absolute row sums.  Over Q(sqrt d) the absolute value of an entry is nu(a + b.sqrt d) = |a| + |b|.sqrt|d| (rd = sqrt|d|): nu is
// submultiplicative and bounds both integer parts of a product.
double denominators_log2(const Dense<QField>& M, const Dense<QField>* B = nullptr) {
  std::vector<int64_t> seen;
  double lg = 0.;
  for (const Dense<QField>* X : {&M, B}) {
    if (!X) continue;
    for (const Rat& e : X->v) {
      if (e.num == 0 || e.den == 1) continue;
      if (std::find(seen.begin(), seen.end(), e.den) != seen.end()) continue;
      seen.push_back(e.den);
      lg += std::log2((double)e.den);
    }
  }
  return lg;
}
double nu(const Dense<QField>& M, const Dense<QField>* B, double rd, size_t i, size_t j) {
  const double a = std::fabs((double)M.at(i, j).num / (double)M.at(i, j).den);
  return B ? a + std::fabs((double)B->at(i, j).num / (double)B->at(i, j).den) * rd : a;
}
std::vector<double> abs_row_sums(const Dense<QField>& M, const Dense<QField>* B = nullptr, double rd = 0.) {
  std::vector<double> s(M.rows, 0.);
  for (size_t i = 0; i < M.rows; ++i)
    for (size_t j = 0; j < M.cols; ++j) s[i] += nu(M, B, rd, i, j);
  return s;
}
// A square root of d modulo the odd prime p, in [1, (p-1)/2]: Tonelli-Shanks.  false when p | d or d is not a square mod p (Euler).
bool sqrt_mod(int64_t d, uint64_t p, int64_t* root) {
  auto mul = [p](uint64_t a, uint64_t b) { return a * b % p; };  // p < 2^32
  auto pw = [&mul](uint64_t b, uint64_t e) { uint64_t r = 1; for (; e; e >>= 1, b = mul(b, b)) if (e & 1) r = mul(r, b); return r; };
  const uint64_t a = (uint64_t)(((d % (int64_t)p) + (int64_t)p) % (int64_t)p);
  if (a == 0 || pw(a, (p - 1) / 2) != 1) return false;
  uint64_t q = p - 1, z = 2;
  int sh = 0;
  while ((q & 1) == 0) { q >>= 1; ++sh; }
  while (pw(z, (p - 1) / 2) != p - 1) ++z;  // a non-residue
  uint64_t c = pw(z, q), t = pw(a, q), r = pw(a, (q + 1) / 2);
  for (int m = sh; t != 1;) {
    int i = 0;
    for (uint64_t u = t; u != 1; u = mul(u, u)) ++i;
    uint64_t b = c;
    for (int e = 0; e < m - i - 1; ++e) b = mul(b, b);
    m = i; c = mul(b, b); t = mul(t, c); r = mul(r, b);
  }
  *root = (int64_t)(r <= p / 2 ? r : p - r);
  return true;
}

// One modular check of `batch` samples through a plan; *bad = number of samples that disagree.
int mmcheck_one_prime(uint64_t p, int bits, uint64_t seed, int batch, int m, int k, int n, const Dense<QField>& L, const plo_csr& vl, const plo_csr& vr,
                      const plo_csr& vp, int* bad) {
  plo_mmcheck_plan* plan = nullptr;
  int rc = plo_mmcheck_plan_create(&plan, (uint32_t)p, m, k, n, (int)L.rows, &vl, &vr, &vp, batch);
  if (rc) return rc;
  int verdict = 0;
  rc = plo_mmcheck_plan_input_bits(plan, bits);
  if (!rc) rc = plo_mmcheck_plan_run(plan, seed, 0, nullptr);
  if (!rc) rc = plo_mmcheck_plan_result(plan, nullptr, nullptr, &verdict);
  plo_mmcheck_plan_destroy(plan);
  *bad = verdict;
  return rc;
}

// fMMchecker / MMchecker on dense rational matrices.
//  modulus > 0: `batch` random evaluations in Z/pZ, p = modulus without its factors of 2 (src/MMchecker.cpp:123-126).
//  modulus == 0: the reference evaluates both sides EXACTLY over Q at a random point with `bitsize`-bit integer coordinates and
//  compares (include/plinopt_library.inl:497-528).  Here: the same test at `batch` random integer points with `bits`-bit coordinates
//  (bits <= 32), decided by residues: with D a common multiple of all denominators, N = D (P.((L ua) o (R ub)) - ua.ub) is an integer
//  vector with |N| <= D (max_o sum_i |P_oi| |L_i|_1 |R_i|_1 + k) 2^(2 bits); the check runs modulo as many word-size primes as it takes
//  for their product to exceed 2 |N|.  All samples agree modulo every prime  =>  N = 0: both sides are EQUAL OVER Q at every point.
//  One sample disagrees modulo one prime => they differ over Q there (no denominator vanishes modulo the primes used).
//  Over Q(sqrt d) (modulus 0, B = the sqrt(d) parts of L, R, P): N = A + B'.sqrt(d) with integers A, B' bounded as above with nu in
//  place of |.| (D over the denominators of both parts).  Only primes where d is a non-zero square are used, each under both
//  embeddings sqrt(d) -> s and -s (same seed and points): if N vanishes under both, 2A = 2B's = 0, so A = B' = 0 mod p.  One
//  embedding alone would not prove it.  *nprimes counts primes, not embeddings.
int mmcheck_dense(uint64_t modulus, int bits, uint64_t seed, int batch, const Dense<QField>& L, const Dense<QField>& R, const Dense<QField>& P, int* nprimes = nullptr,
                  int64_t d = 0, const Dense<QField>* B = nullptr) {
  int m, k, n;
  plo_LRP2MM((int)L.cols, (int)R.cols, (int)P.rows, &m, &k, &n);
  if (L.rows != R.rows || L.rows != P.cols) return 2;                                                   // MMchecker.cpp:65-71
  if ((int)L.cols != m * k || (int)R.cols != k * n || (int)P.rows != m * n) return 3;                  // library.inl:487-495
  if (bits < 1) bits = 1;
  if (bits > 32) bits = 32;
  uint64_t p = modulus;
  if (p > 0) { while ((p % 2) == 0) p >>= 1; if (p == 1) p = 2; }                                      // MMchecker.cpp:123-126
  CsrHost cl, cr, cp;
  const Dense<QField>* Lb = B ? &B[0] : nullptr;
  const Dense<QField>* Rb = B ? &B[1] : nullptr;
  const Dense<QField>* Pb = B ? &B[2] : nullptr;
  const SparseQ sL(L, Lb), sR(R, Rb), sP(P, Pb);
  if (p > 0) {
    if (p >= (1ull << 32)) { plo::set_error("mmchecker: modulus must be below 2^32 after stripping factors of 2"); return PLO_E_ARG; }
    if (!(to_csr(sL, (int64_t)p, cl) && to_csr(sR, (int64_t)p, cr) && to_csr(sP, (int64_t)p, cp))) {
      plo::set_error("mmchecker: a denominator is not invertible modulo %llu", (unsigned long long)p);
      return PLO_E_ARG;
    }
    int bad = 0;
    const int rc = mmcheck_one_prime(p, bits, seed, batch, m, k, n, L, cl.view((int)L.rows, (int)L.cols), cr.view((int)R.rows, (int)R.cols), cp.view((int)P.rows, (int)P.cols), &bad);
    if (nprimes) *nprimes = 1;
    return rc ? rc : bad;
  }
  // over Q or Q(sqrt d): size of the integer N above
  const double rd = std::sqrt(std::fabs((double)d));
  const std::vector<double> sl = abs_row_sums(L, Lb, rd), sr = abs_row_sums(R, Rb, rd);
  double worst = 0.;
  for (size_t o = 0; o < P.rows; ++o) {
    double t = 0.;
    for (size_t i = 0; i < P.cols; ++i) { const double v = nu(P, Pb, rd, o, i); if (v != 0.) t += v * sl[i] * sr[i]; }
    worst = std::max(worst, t);
  }
  const double need = denominators_log2(L, Lb) + denominators_log2(R, Rb) + denominators_log2(P, Pb) + std::log2(worst + (double)k + 1.) + 2. * bits + 3.;  // + sign, rounding slack
  double have = 0.;
  int used = 0;
  for (p = 2147483647ull; p > (1ull << 30) && have <= need; p -= 2) {
    if (!is_prime(p)) continue;
    int64_t s = 0;
    if (B && !sqrt_mod(d, p, &s)) continue;  // over Q(sqrt d): p | d, or d is not a square mod p
    auto image = [&](int64_t root) { return to_csr(sL, (int64_t)p, cl, root) && to_csr(sR, (int64_t)p, cr, root) && to_csr(sP, (int64_t)p, cp, root); };
    if (!image(s)) continue;  // a denominator vanishes (under every embedding): next prime
    int bad = 0;
    for (int e = 0; e < (B ? 2 : 1) && !bad; ++e) {
      if (e) image((int64_t)p - s);
      const int rc = mmcheck_one_prime(p, bits, seed, batch, m, k, n, L, cl.view((int)L.rows, (int)L.cols), cr.view((int)R.rows, (int)R.cols), cp.view((int)P.rows, (int)P.cols), &bad);
      if (rc) return rc;
    }
    ++used;
    if (nprimes) *nprimes = used;
    if (bad) return 1;
    have += std::log2((double)p);
  }
  if (have <= need) { plo::set_error("mmchecker: ran out of primes"); return PLO_E_RANGE; }
  return 0;
}

}  // namespace

// Factorizer  include/plinopt_sparsify.inl:924-990.  F = field of the search (Q or Z/qZ).
template <class F>
static int run_factorizer(const F& f, int rows, int cols, const int64_t* num, const int64_t* den, int innerdim,
                          uint64_t loops, uint64_t seed, int64_t* alt_num, int64_t* alt_den, int64_t* cob_num, int64_t* cob_den, uint64_t* report) {
  typedef Dense<F> Mat;
  const size_t r = (size_t)rows, n = (size_t)cols;
  const size_t k = innerdim == 0 ? n : (size_t)innerdim;  // in [n, r]: checked by plo_factorizer
  const Mat M = load(f, r, n, num, den);
  FactorHost<F> fh(f);
  Sparsifier<F> la(f, nullptr);
  Mat Alt(f, r, k), CoB(f, k, n);
  const auto sc = fh.nonzeroes(M);
  Tricounter nbops{sc.first, sc.second, n};  // "Start with M and Identity" :958
  uint64_t windex = PLO_NO_INDEX;
  if (r == n) {  // :945-951 identity factorization
    CoB = M;
    for (size_t i = 0; i < r; ++i) Alt.at(i, i) = f.one();
  } else {
    for (size_t i = 0; i < r; ++i) for (size_t j = 0; j < n; ++j) Alt.at(i, j) = M.at(i, j);  // sparse2sparse(Alt, M) :953
    for (size_t i = 0; i < n; ++i) CoB.at(i, i) = f.one();
    if (la.rank(M) != n) { plo::set_error("plo_factorizer: the matrix has not full column rank (backSolver precondition, :754)"); return PLO_E_ARG; }
    // modulus of the device search: q itself, or a 31-bit prime for rational input (scores are re-derived exactly below)
    const uint32_t qprimes[3] = {2147483647u, 2147483629u, 2147483587u};
    const int tries = F::modular ? 1 : 3;
    bool done = false;
    for (int attempt = 0; attempt < tries && !done; ++attempt) {
      const uint32_t p = F::modular ? (uint32_t)f.characteristic() : qprimes[attempt];
      ZpField Z((int64_t)p);
      std::vector<uint32_t> res(r * n);
      bool invertible = true;
      for (size_t e = 0; e < r * n && invertible; ++e) {
        const int64_t d = den ? den[e] : 1;
        if (Z.canon(d) == 0) { invertible = false; break; }
        res[e] = (uint32_t)Z.div(Z.canon(num[e]), Z.canon(d));
      }
      if (!invertible) {
        if (F::modular) { plo::set_error("plo_factorizer: a denominator is not invertible modulo %u", p); return PLO_E_ARG; }
        continue;
      }
      plo_factor_best best;
      const int rc = plo_factor_sweep(p, rows, cols, (int)k, res.data(), seed, 0, loops, &best, nullptr);
      if (rc) return rc;
      done = true;
      if (best.index == PLO_NO_INDEX) break;
      const Tricounter gpu{best.nnz_alt, best.nno_alt, best.nnz_cob};
      if (!tricOpCount(gpu, nbops)) break;  // nothing beats M = M.I  (:968)
      std::vector<int32_t> order32(r);
      plo_factor_decode(rows, seed, best.index, order32.data());
      Mat lAlt, lCoB;
      Tricounter exact{0, 0, 0};
      const bool ok = fh.backSolver(lCoB, lAlt, M, k, std::vector<int>(order32.begin(), order32.end()), exact);
      if (!ok || exact != gpu) { done = false; continue; }  // a residue vanished modulo p by accident: search again with another prime
      nbops = exact; Alt = lAlt; CoB = lCoB; windex = best.index;
    }
    if (!done) { plo::set_error("plo_factorizer: the modular scores disagreed with the exact ones for every prime tried"); return PLO_E_RANGE; }
  }
  store(Alt, alt_num, alt_den);
  store(CoB, cob_num, cob_den);
  if (report) {
    report[0] = sc.first; report[1] = sc.second; report[2] = n;
    report[3] = nbops[0]; report[4] = nbops[1]; report[5] = nbops[2];
    report[6] = windex; report[7] = la.consistency(M, Alt, CoB) ? 1 : 0;
  }
  return PLO_OK;
}

// Orbit action on a triple (src/orbiter.cpp:284-294) without the Kronecker products:
// row l of L.(U^-1 (x) V) = vec(U^-T A_l V), of R.(V^-T (x) W) = vec(V^-1 B_l W); column l of (U (x) W^-1).P = vec(U C_l W^-T)
template <class F>
static void orbit_transform(const F& f, int m, int k, int n, int r, const Dense<F>& L, const Dense<F>& R, const Dense<F>& P,
                            const std::vector<int32_t>& U, const std::vector<int32_t>& V, const std::vector<int32_t>& W,
                            Dense<F>& Lj, Dense<F>& Rg, Dense<F>& hP) {
  Sparsifier<F> la(f, nullptr);
  auto tomat = [&](const std::vector<int32_t>& a, int s) {
    Dense<F> M(f, (size_t)s, (size_t)s);
    for (size_t e = 0; e < a.size(); ++e) M.v[e] = f.from_ratio(a[e], 1);
    return M;
  };
  const Dense<F> Um = tomat(U, m), Vm = tomat(V, k), Wm = tomat(W, n);
  const Dense<F> iU = la.inverse(Um), iV = la.inverse(Vm), iW = la.inverse(Wm);
  const Dense<F> iUT = la.transpose(iU), iWT = la.transpose(iW);
  for (int l = 0; l < r; ++l) {
    Dense<F> A(f, (size_t)m, (size_t)k), B(f, (size_t)k, (size_t)n), C(f, (size_t)m, (size_t)n);
    for (int e = 0; e < m * k; ++e) A.v[e] = L.at((size_t)l, (size_t)e);
    for (int e = 0; e < k * n; ++e) B.v[e] = R.at((size_t)l, (size_t)e);
    for (int e = 0; e < m * n; ++e) C.v[e] = P.at((size_t)e, (size_t)l);
    const Dense<F> Y1 = la.mul(la.mul(iUT, A), Vm), Y2 = la.mul(la.mul(iV, B), Wm), Y3 = la.mul(la.mul(Um, C), iWT);
    for (int e = 0; e < m * k; ++e) Lj.at((size_t)l, (size_t)e) = Y1.v[e];
    for (int e = 0; e < k * n; ++e) Rg.at((size_t)l, (size_t)e) = Y2.v[e];
    for (int e = 0; e < m * n; ++e) hP.at((size_t)e, (size_t)l) = Y3.v[e];
  }
}

static int g_sweep_devices = 1;  // devices a host-level sweep is sharded over (plo_set_sweep_devices)

static inline int64_t store_one(const ZpField& f, int64_t e) { return f.canon(e); }
static inline int64_t store_one(const QField&, const Rat&) { return 0; }
static inline int64_t num_of(const Rat& e) { return e.num; }
static inline int64_t den_of(const Rat& e) { return e.den; }
static inline int64_t num_of(int64_t e) { return e; }
static inline int64_t den_of(int64_t) { return 1; }
// Depender  src/dependency.cpp:106-169 over the field F.
template <class F>
static int run_depender(const F& f, const Dense<QField>& B, const std::vector<Rat>& user, size_t maxnumcoeff, int level, uint64_t max_hits,
                        plo_dep_hit* hits, uint64_t* nhits, uint64_t* ncand, char* text, size_t text_cap, size_t* text_len,
                        int64_t* coef_num, int64_t* coef_den, int* ncoef) {
  typedef typename F::Elt Elt;
  const size_t r = B.rows, n = B.cols;
  Dense<F> M(f, r, n);
  for (size_t e = 0; e < B.v.size(); ++e) M.v[e] = f.from_ratio(B.v[e].num, B.v[e].den);
  const std::vector<Elt> C = field_coefficients(f, dependency_coefficients(B, user, maxnumcoeff));
  const size_t c = C.size();
  if (ncoef) *ncoef = (int)c;
  if (coef_num) {
    Dense<F> tmp(f, 1, c);
    for (size_t v = 0; v < c; ++v) tmp.v[v] = C[v];
    store(tmp, coef_num, coef_den);
  }
  if (c == 0 || level < 2) { if (nhits) *nhits = 0; if (ncand) *ncand = 0; if (text_len) *text_len = 0; return PLO_OK; }
  // tables in the field: residues, or integers scaled by the common denominator D
  std::vector<int64_t> base(r * n), prod(r * c * n);
  uint32_t p = 0;
  if (F::modular) {
    p = (uint32_t)f.characteristic();
    for (size_t e = 0; e < r * n; ++e) base[e] = store_one(f, M.v[e]);
    for (size_t q = 0; q < r; ++q) for (size_t v = 0; v < c; ++v) for (size_t j = 0; j < n; ++j) prod[(q * c + v) * n + j] = store_one(f, f.mul(C[v], M.at(q, j)));
  } else {
    std::vector<Elt> pe(r * c * n);
    for (size_t q = 0; q < r; ++q) for (size_t v = 0; v < c; ++v) for (size_t j = 0; j < n; ++j) pe[(q * c + v) * n + j] = f.mul(C[v], M.at(q, j));
    wide D = 1;
    auto fold = [&D](int64_t den) { D = D / wgcd(D, den) * den; if (D > ((wide)1 << 60)) throw RangeError("common denominator exceeds 60 bits"); };
    for (const Elt& e : M.v) fold(den_of(e));
    for (const Elt& e : pe) fold(den_of(e));
    auto scale = [&D](const Elt& e) { const wide v = (wide)num_of(e) * (D / den_of(e)); if (wabs(v) > ((wide)1 << 60)) throw RangeError("scaled entry exceeds 60 bits"); return (int64_t)v; };
    for (size_t e = 0; e < r * n; ++e) base[e] = scale(M.v[e]);
    for (size_t e = 0; e < pe.size(); ++e) prod[e] = scale(pe[e]);
  }
  uint64_t found = 0;
  const int rc = plo_dependency_explore(p, (int)r, (int)n, (int)c, level, base.data(), prod.data(), max_hits, hits, &found, ncand);
  if (nhits) *nhits = found;  // also set with PLO_E_RANGE: the number of records the caller has to make room for
  if (rc) return rc;
  if (text) {
    DependencyHost<F> dh(f);
    std::string all;
    const uint64_t stored = found < max_hits ? found : max_hits;
    for (uint64_t h = 0; h < stored; ++h) { all += dh.line(M, C, hits[h]); all += '\n'; }
    const size_t len = all.size() < text_cap ? all.size() : (text_cap ? text_cap - 1 : 0);
    memcpy(text, all.data(), len);
    if (text_cap) text[len] = 0;
    if (text_len) *text_len = all.size();
  }
  return PLO_OK;
}

namespace plo {
int quad_field_ok(int64_t d, int measure, const char* who);  // orbit_sweep.cu: X^2 - d defines a field, G2 has a real embedding
// orbit_sweep.cu: the sweep of [lo,hi) sharded over `ndev` devices, `create` making the plan on each
int orbit_sweep_sharded(int ndev, int measure, uint64_t lo, uint64_t hi, plo_orbit_best* best, const std::function<int(plo_orbit_plan**)>& create);
}

namespace {
// A triple over Q (B empty), or over Q(sqrt d): entry a + b.sqrt(d) with a in L, R, P and b in B[0], B[1], B[2].
struct FieldTriple {
  int64_t d = 0;
  Dense<QField> L, R, P;
  std::vector<Dense<QField>> B;
  const Dense<QField>* surds() const { return B.empty() ? nullptr : B.data(); }
  int r() const { return (int)L.rows; }
  void count(uint32_t& nnz, uint32_t& nno) const {
    const Dense<QField>* b = surds();
    count_nonzeroes(L, nnz, nno, b ? &b[0] : nullptr); count_nonzeroes(R, nnz, nno, b ? &b[1] : nullptr); count_nonzeroes(P, nnz, nno, b ? &b[2] : nullptr);
  }
  double g2() const { return growth_G2(L, R, P, surds(), B.empty() ? 0. : std::sqrt((double)d)); }
  // the orbit action is Q-linear with integer factors: over Q(sqrt d) each part transforms on its own
  FieldTriple transformed(int m, int k, int n, const std::vector<int32_t>& U, const std::vector<int32_t>& V, const std::vector<int32_t>& W) const {
    QField Q;
    FieldTriple o = *this;
    orbit_transform(Q, m, k, n, r(), L, R, P, U, V, W, o.L, o.R, o.P);
    if (!B.empty()) orbit_transform(Q, m, k, n, r(), B[0], B[1], B[2], U, V, W, o.B[0], o.B[1], o.B[2]);
    return o;
  }
  int mmcheck(int bits, uint64_t seed, int batch) const { return mmcheck_dense(0, bits, seed, batch, L, R, P, nullptr, d, surds()); }
};
// The arrays of a triple at the C ABI: (an, ad, bn, bd) for each of L, R, P, entry e of a matrix being an[e]/ad[e] + bn[e]/bd[e].sqrt(d).
// Over Q the sqrt(d) parts bn, bd are NULL; NULL denominators mean 1.
FieldTriple load_triple(int64_t d, int Lrows, int Lcols, int Rrows, int Rcols, int Prows, int Pcols, const int64_t* const q[12]) {
  QField Q;
  FieldTriple t;
  t.L = load(Q, (size_t)Lrows, (size_t)Lcols, q[0], q[1]); t.R = load(Q, (size_t)Rrows, (size_t)Rcols, q[4], q[5]); t.P = load(Q, (size_t)Prows, (size_t)Pcols, q[8], q[9]);
  if (!q[2]) return t;
  t.d = d;
  t.B = {load(Q, (size_t)Lrows, (size_t)Lcols, q[2], q[3]), load(Q, (size_t)Rrows, (size_t)Rcols, q[6], q[7]), load(Q, (size_t)Prows, (size_t)Pcols, q[10], q[11])};
  return t;
}
void store_triple(const FieldTriple& t, int64_t* const q[12]) {
  store(t.L, q[0], q[1]); store(t.R, q[4], q[5]); store(t.P, q[8], q[9]);
  for (int x = 0; x < (int)t.B.size(); ++x) store(t.B[(size_t)x], q[4 * x + 2], q[4 * x + 3]);
}

// integer images of a rational triple (every entry times the matrix' common LCD) and the sweep entry point that fits them
struct OrbitImages {
  std::vector<int64_t> L64, R64, P64;
  int64_t dl = 1, dr = 1, dp = 1;
  bool fits32 = true;
  explicit OrbitImages(const FieldTriple& t) {
    auto split = [](const Dense<QField>& M, std::vector<int64_t>& n, std::vector<int64_t>& d) {
      n.resize(M.v.size()); d.resize(M.v.size());
      for (size_t e = 0; e < M.v.size(); ++e) { n[e] = M.v[e].num; d[e] = M.v[e].den; }
    };
    std::vector<int64_t> ln, ld, rn, rd, pn, pd;
    split(t.L, ln, ld); split(t.R, rn, rd); split(t.P, pn, pd);
    const wide lim = (wide)1 << 46;
    dl = lcd_of(ld.data(), ld.size(), lim); dr = lcd_of(rd.data(), rd.size(), lim); dp = lcd_of(pd.data(), pd.size(), lim);
    L64 = scale_int64(ln.data(), ld.data(), ln.size(), dl, fits32);
    R64 = scale_int64(rn.data(), rd.data(), rn.size(), dr, fits32);
    P64 = scale_int64(pn.data(), pd.data(), pn.size(), dp, fits32);
  }
  int sweep(int m, int k, int n, int r, int measure, int mode, uint64_t seed, uint64_t lo, uint64_t hi, plo_orbit_best* best) const {
    if (fits32) {
      const std::vector<int32_t> Li(L64.begin(), L64.end()), Ri(R64.begin(), R64.end()), Pi(P64.begin(), P64.end());
      return plo_orbit_sweep_devices(g_sweep_devices, m, k, n, r, Li.data(), Ri.data(), Pi.data(), (int32_t)dl, (int32_t)dr, (int32_t)dp, measure, mode, seed, lo, hi, best);
    }
    // common denominators beyond 2^31 (2x2x2_7_DPS-intermediate-12.0695): the 64-bit input path
    return plo_orbit_sweep64(m, k, n, r, L64.data(), R64.data(), P64.data(), dl, dr, dp, measure, mode, seed, lo, hi, best);
  }
};
// The same over Q(sqrt d): both integer parts of each matrix over one common denominator (plo_orbit_plan_create_quad)
struct QuadOrbitImages {
  int64_t d;
  std::vector<int64_t> part[6];  // La, Lb, Ra, Rb, Pa, Pb
  int64_t den[3];
  explicit QuadOrbitImages(const FieldTriple& t) : d(t.d) {
    const Dense<QField>* M[6] = {&t.L, &t.B[0], &t.R, &t.B[1], &t.P, &t.B[2]};
    bool fits32 = true;  // the plan picks its own storage
    for (int x = 0; x < 3; ++x) {
      std::vector<int64_t> num[2], dd[2], all;
      for (int h = 0; h < 2; ++h)
        for (const Rat& e : M[2 * x + h]->v) { num[h].push_back(e.num); dd[h].push_back(e.den); all.push_back(e.den); }
      den[x] = lcd_of(all.data(), all.size(), (wide)1 << 46);
      for (int h = 0; h < 2; ++h) part[2 * x + h] = scale_int64(num[h].data(), dd[h].data(), num[h].size(), den[x], fits32);
    }
  }
  int sweep(int m, int k, int n, int r, int measure, int mode, uint64_t seed, uint64_t lo, uint64_t hi, plo_orbit_best* best) const {
    return plo::orbit_sweep_sharded(g_sweep_devices, measure, lo, hi, best, [&](plo_orbit_plan** pl) {
      return plo_orbit_plan_create_quad(pl, d, m, k, n, r, part[0].data(), part[1].data(), part[2].data(), part[3].data(), part[4].data(), part[5].data(),
                                        den[0], den[1], den[2], measure, mode, seed);
    });
  }
};
bool orbit_improves(int measure, const plo_orbit_best& b, double init_score, uint32_t init_nnz, uint32_t init_nno) {  // src/orbiter.cpp:300-302, 330-331
  if (b.index == PLO_NO_INDEX) return false;
  if (measure == PLO_MEASURE_G2) return b.score < init_score * (1.0 - 1e-12);  // beyond the rounding of the two evaluations
  return b.nnz < init_nnz || (b.nnz == init_nnz && b.nno < init_nno);
}

// The '# Found opt:' records of src/orbiter.cpp:300-318 made deterministic: the reference prints every candidate that improves
// on the best so far as its threads meet them; in index order those are the successive minima of the prefixes [0, i] that also
// improve on the input.  They are found backwards: the winner of [0, loops), then the winner of [0, its index), and so on
// (each sweep is shorter; about twice the cost of one sweep in total).  records come back in increasing index order.
// The body of plo_orbiter_progress over Q (OrbitImages) and over Q(sqrt d) (QuadOrbitImages) after their argument checks; q as in load_triple.
template <class Images>
int orbiter_progress(const char* who, int64_t d, int r, int Lcols, int Rcols, int Prows, const int64_t* const q[12], int measure, int mode,
                     uint64_t seed, uint64_t loops, uint64_t capacity, plo_orbit_best* records, uint64_t* count) {
  int m, k, n;
  if (const int rc = plo::check_device()) return rc;
  if (const int rc = mm_shape(who, Lcols, Rcols, Prows, &m, &k, &n)) return rc;
  return guarded(who, [&] {
    const FieldTriple in = load_triple(d, r, Lcols, r, Rcols, Prows, r, q);
    uint32_t init_nnz = 0, init_nno = 0;
    in.count(init_nnz, init_nno);
    const double init_score = measure == PLO_MEASURE_G2 ? in.g2() : (double)init_nnz;
    const Images img(in);
    std::vector<plo_orbit_best> rev;
    uint64_t hi = loops;
    while (hi > 0 && rev.size() < 256) {
      plo_orbit_best b;
      const int rc = img.sweep(m, k, n, r, measure, mode, seed, 0, hi, &b);
      if (rc) return rc;
      if (!orbit_improves(measure, b, init_score, init_nnz, init_nno)) break;
      rev.push_back(b);
      hi = b.index;
    }
    *count = rev.size();
    if (rev.size() > capacity) { plo::set_error("%s: %zu records, room for %llu", who, rev.size(), (unsigned long long)capacity); return PLO_E_RANGE; }
    for (size_t t = 0; t < rev.size(); ++t) records[t] = rev[rev.size() - 1 - t];
    return PLO_OK;
  });
}

// Orbiter src/orbiter.cpp:215-360: the sweep, the acceptance against the input (:330-331), the exact transform of the winner and
// the MMchecker of the returned triple (:355).  The body of plo_orbiter over Q (OrbitImages) and over Q(sqrt d) (QuadOrbitImages)
// after their argument checks; q in, o out, both as in load_triple.
template <class Images>
int orbiter(const char* who, int64_t d, int r, int Lcols, int Rcols, int Prows, const int64_t* const q[12], int measure, int mode, uint64_t seed,
            uint64_t loops, int64_t* const o[12], plo_orbiter_report* rep) {
  int m, k, n;
  if (const int rc = plo::check_device()) return rc;
  if (const int rc = mm_shape(who, Lcols, Rcols, Prows, &m, &k, &n)) return rc;
  return guarded(who, [&] {
    const FieldTriple in = load_triple(d, r, Lcols, r, Rcols, Prows, r, q);
    memset(rep, 0, sizeof(*rep));
    rep->m = m; rep->k = k; rep->n = n;
    in.count(rep->init_nnz, rep->init_nno);
    rep->init_score = measure == PLO_MEASURE_G2 ? in.g2() : (double)rep->init_nnz;
    const Images img(in);
    const int rc = img.sweep(m, k, n, r, measure, mode, seed, 0, loops, &rep->best);
    if (rc) return rc;
    const bool improved = orbit_improves(measure, rep->best, rep->init_score, rep->init_nnz, rep->init_nno);
    FieldTriple out;
    if (improved) {
      std::vector<int32_t> U((size_t)m * m), V((size_t)k * k), W((size_t)n * n);
      plo_orbit_decode(m, k, n, mode, seed, rep->best.index, U.data(), V.data(), W.data());
      out = in.transformed(m, k, n, U, V, W);
    } else {
      out = in;
    }
    rep->improved = improved ? 1 : 0;
    rep->mm_verdict = out.mmcheck(32, seed ^ 0x4D4D636865636Bull, 32);
    store_triple(out, o);
    return PLO_OK;
  });
}

// fMMchecker (src/MMchecker.cpp:48-81) of a loaded triple: the counts, 2 on an inner dimension mismatch, then the device and the check
int mmchecker_triple(const FieldTriple& t, uint64_t modulus, int bits, uint64_t seed, int batch, uint32_t* nnz_nno, int* nprimes) {
  if (nnz_nno) { nnz_nno[0] = nnz_nno[1] = 0; t.count(nnz_nno[0], nnz_nno[1]); }
  if (nprimes) *nprimes = 0;
  if (t.L.rows != t.R.rows || t.L.rows != t.P.cols) return 2;
  const int rc = plo::check_device();
  return rc ? rc : mmcheck_dense(modulus, bits, seed, batch, t.L, t.R, t.P, nprimes, t.d, t.surds());
}
}  // namespace

extern "C" {

void plo_LRP2MM(int Lcols, int Rcols, int Prows, int* m, int* k, int* n) {
  const size_t nn = (size_t)std::sqrt((double)((size_t)Rcols * (size_t)Prows / (size_t)(Lcols ? Lcols : 1)));
  *n = (int)nn;
  *m = nn ? (int)((size_t)Prows / nn) : 0;
  *k = nn ? (int)((size_t)Rcols / nn) : 0;
}

struct plo_slp_matrix_impl { plo::host::SparseRows M; };

int plo_slp_build(const char* text, char outchar, plo_slp_matrix** out, int* rows, int* cols, int64_t* nnz) {
  if (!text || !out) { plo::set_error("plo_slp_build: bad argument"); return PLO_E_ARG; }
  try {
    plo::host::SlpBuilder b;
    plo_slp_matrix_impl* h = new plo_slp_matrix_impl();
    h->M = b.build(text, outchar ? outchar : 'o');
    *out = reinterpret_cast<plo_slp_matrix*>(h);
    if (rows) *rows = (int)h->M.rows;
    if (cols) *cols = (int)h->M.cols;
    if (nnz) *nnz = (int64_t)h->M.nnz();
    return PLO_OK;
  } catch (const std::exception& e) {
    plo::set_error("plo_slp_build: %s", e.what());
    return PLO_E_RANGE;
  }
}
int plo_slp_export(const plo_slp_matrix* m, int64_t* ptr, int32_t* col, int64_t* num, int64_t* den) {
  if (!m || !ptr || !col || !num || !den) { plo::set_error("plo_slp_export: bad argument"); return PLO_E_ARG; }
  const plo::host::SparseRows& M = reinterpret_cast<const plo_slp_matrix_impl*>(m)->M;
  int64_t t = 0;
  ptr[0] = 0;
  for (size_t i = 0; i < M.rows; ++i) {
    for (const auto& e : M.r[i]) { col[t] = e.first; num[t] = e.second.num; den[t] = e.second.den; ++t; }
    ptr[i + 1] = t;
  }
  return PLO_OK;
}
void plo_slp_free(plo_slp_matrix* m) { delete reinterpret_cast<plo_slp_matrix_impl*>(m); }

int plo_sparsifier(uint64_t q, int rows, int cols, const int64_t* num, const int64_t* den, int blocksize,
                   int maxnumcoeff, int initialElimination, int64_t* cob_num, int64_t* cob_den,
                   int64_t* res_num, int64_t* res_den, int* consistent, uint64_t* stats, int log_fd) {
  if (!num || !cob_num || !res_num || rows < 1 || cols < 1 || blocksize < 0 || maxnumcoeff < 1 || q >= (1ull << 32)) {
    plo::set_error("plo_sparsifier: bad argument");
    return PLO_E_ARG;
  }
  int rc = plo::check_device();
  if (rc) return rc;
  FdBuf buf(log_fd);
  std::ostream logstream(&buf);
  std::ostream* log = log_fd >= 0 ? &logstream : nullptr;
  return guarded("plo_sparsifier", [&] {
    if (q == 0) { QField f; return run_sparsifier(f, rows, cols, num, den, blocksize, maxnumcoeff, initialElimination, cob_num, cob_den, res_num, res_den, consistent, stats, log); }
    ZpField f((int64_t)q);
    return run_sparsifier(f, rows, cols, num, den, blocksize, maxnumcoeff, initialElimination, cob_num, cob_den, res_num, res_den, consistent, stats, log);
  });
}

int plo_orbiter_progress(int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                         const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd, const int64_t* Pn,
                         const int64_t* Pd, uint64_t capacity, plo_orbit_best* records, uint64_t* count) {
  if (!Ln || !Rn || !Pn || !records || !count || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) { plo::set_error("plo_orbiter_progress: bad argument"); return PLO_E_ARG; }
  const int64_t* const q[12] = {Ln, Ld, nullptr, nullptr, Rn, Rd, nullptr, nullptr, Pn, Pd, nullptr, nullptr};
  return orbiter_progress<OrbitImages>("plo_orbiter_progress", 0, r, Lcols, Rcols, Prows, q, measure, mode, seed, loops, capacity, records, count);
}

int plo_orbiter(int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd, const int64_t* Pn,
                const int64_t* Pd, int64_t* oLn, int64_t* oLd, int64_t* oRn, int64_t* oRd, int64_t* oPn, int64_t* oPd,
                plo_orbiter_report* rep) {
  if (!Ln || !Rn || !Pn || !oLn || !oRn || !oPn || !oLd || !oRd || !oPd || !rep || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) {
    plo::set_error("plo_orbiter: bad argument");
    return PLO_E_ARG;
  }
  const int64_t* const q[12] = {Ln, Ld, nullptr, nullptr, Rn, Rd, nullptr, nullptr, Pn, Pd, nullptr, nullptr};
  int64_t* const o[12] = {oLn, oLd, nullptr, nullptr, oRn, oRd, nullptr, nullptr, oPn, oPd, nullptr, nullptr};
  return orbiter<OrbitImages>("plo_orbiter", 0, r, Lcols, Rcols, Prows, q, measure, mode, seed, loops, o, rep);
}

// The same two drivers over Q(sqrt d) (`orbiter -P "X^2-d"`): pair layout (an, ad, bn, bd) per matrix, inputs and outputs.
int plo_orbiter_progress_quad(int64_t d, int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                              const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn, const int64_t* Lbd, const int64_t* Ran,
                              const int64_t* Rad, const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan, const int64_t* Pad,
                              const int64_t* Pbn, const int64_t* Pbd, uint64_t capacity, plo_orbit_best* records, uint64_t* count) {
  if (!Lan || !Lbn || !Ran || !Rbn || !Pan || !Pbn || !records || !count || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1 ||
      (measure != PLO_MEASURE_NNZ && measure != PLO_MEASURE_G2)) {
    plo::set_error("plo_orbiter_progress_quad: bad argument");
    return PLO_E_ARG;
  }
  if (const int rc = plo::quad_field_ok(d, measure, "plo_orbiter_progress_quad")) return rc;
  const int64_t* const q[12] = {Lan, Lad, Lbn, Lbd, Ran, Rad, Rbn, Rbd, Pan, Pad, Pbn, Pbd};
  return orbiter_progress<QuadOrbitImages>("plo_orbiter_progress_quad", d, r, Lcols, Rcols, Prows, q, measure, mode, seed, loops, capacity, records, count);
}

int plo_orbiter_quad(int64_t d, int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                     const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn, const int64_t* Lbd, const int64_t* Ran, const int64_t* Rad,
                     const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan, const int64_t* Pad, const int64_t* Pbn, const int64_t* Pbd,
                     int64_t* oLan, int64_t* oLad, int64_t* oLbn, int64_t* oLbd, int64_t* oRan, int64_t* oRad, int64_t* oRbn, int64_t* oRbd,
                     int64_t* oPan, int64_t* oPad, int64_t* oPbn, int64_t* oPbd, plo_orbiter_report* rep) {
  int64_t* const o[12] = {oLan, oLad, oLbn, oLbd, oRan, oRad, oRbn, oRbd, oPan, oPad, oPbn, oPbd};
  if (!Lan || !Lbn || !Ran || !Rbn || !Pan || !Pbn || std::find(o, o + 12, nullptr) != o + 12 || !rep || r < 1 || Lcols < 1 || Rcols < 1 ||
      Prows < 1 || (measure != PLO_MEASURE_NNZ && measure != PLO_MEASURE_G2)) {
    plo::set_error("plo_orbiter_quad: bad argument");
    return PLO_E_ARG;
  }
  if (const int rc = plo::quad_field_ok(d, measure, "plo_orbiter_quad")) return rc;
  const int64_t* const q[12] = {Lan, Lad, Lbn, Lbd, Ran, Rad, Rbn, Rbd, Pan, Pad, Pbn, Pbd};
  return orbiter<QuadOrbitImages>("plo_orbiter_quad", d, r, Lcols, Rcols, Prows, q, measure, mode, seed, loops, o, rep);
}

int plo_factorizer(uint64_t q, int rows, int cols, const int64_t* num, const int64_t* den, int innerdim, uint64_t loops, uint64_t seed,
                   int64_t* alt_num, int64_t* alt_den, int64_t* cob_num, int64_t* cob_den, uint64_t* report) {
  if (!num || !alt_num || !cob_num || rows < 1 || cols < 1 || innerdim < 0) { plo::set_error("plo_factorizer: bad argument"); return PLO_E_ARG; }
  const int k = innerdim == 0 ? cols : innerdim;
  if (k > rows || k < cols) {  // :936-942, before any other shape check, as the reference: a wide matrix is refused here
    plo::set_error("Fail: inner dimension has to be between %d and %d.", cols, rows);
    return -1;
  }
  if (rows != cols && (cols > 64 || rows > 512)) {
    plo::set_error("plo_factorizer: the device search takes at most 64 columns and 512 rows (got %d x %d)", rows, cols);
    return PLO_E_SHAPE;
  }
  return guarded("plo_factorizer", [&] {
    if (q == 0) { QField Q; return run_factorizer(Q, rows, cols, num, den, innerdim, loops, seed, alt_num, alt_den, cob_num, cob_den, report); }
    uint64_t p = q;
    while ((p % 2) == 0) p >>= 1;
    if (p < 3 || p >= (1ull << 31) || !is_prime(p)) { plo::set_error("plo_factorizer: the modulus must be an odd prime below 2^31"); return PLO_E_ARG; }
    ZpField Z((int64_t)p);
    return run_factorizer(Z, rows, cols, num, den, innerdim, loops, seed, alt_num, alt_den, cob_num, cob_den, report);
  });
}

int plo_depender(uint64_t q, int rows, int cols, const int64_t* num, const int64_t* den, int nuser, const int64_t* user_num,
                 const int64_t* user_den, int maxnumcoeff, int level, uint64_t max_hits, plo_dep_hit* hits, uint64_t* nhits,
                 uint64_t* ncand, char* text, uint64_t text_cap, uint64_t* text_len, int64_t* coef_num, int64_t* coef_den, int* ncoef) {
  if (!num || rows < 1 || cols < 1 || maxnumcoeff < 1 || level < 1 || (max_hits && !hits) || (nuser > 0 && !user_num)) {
    plo::set_error("plo_depender: bad argument");
    return PLO_E_ARG;
  }
  return guarded("plo_depender", [&] {
    QField Q;
    const Dense<QField> B = load(Q, (size_t)rows, (size_t)cols, num, den);
    std::vector<Rat> user;
    for (int u = 0; u < nuser; ++u) user.push_back(Rat::make(user_num[u], user_den ? user_den[u] : 1));
    size_t tl = 0;
    int rc;
    if (q == 0) rc = run_depender(Q, B, user, (size_t)maxnumcoeff, level, max_hits, hits, nhits, ncand, text, (size_t)text_cap, &tl, coef_num, coef_den, ncoef);
    else {
      if (q >= (1ull << 32) || !is_prime(q)) { plo::set_error("plo_depender: the modulus must be a prime below 2^32"); return PLO_E_ARG; }
      ZpField Z((int64_t)q);
      rc = run_depender(Z, B, user, (size_t)maxnumcoeff, level, max_hits, hits, nhits, ncand, text, (size_t)text_cap, &tl, coef_num, coef_den, ncoef);
    }
    if (text_len) *text_len = tl;
    return rc;
  });
}

// Orbiter over Z/qZ (`orbiter -m q`, src/orbiter.cpp:419-426 -> Orbiter<0>()(QQ, F, ...)): the matrices are reduced
// modulo q first (:232-234) and the whole search, the acceptance (:330-331) and the final check run in the field.
int plo_orbiter_modp(uint64_t q, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows, const int64_t* Ln,
                     const int64_t* Ld, const int64_t* Rn, const int64_t* Rd, const int64_t* Pn, const int64_t* Pd, int64_t* oL,
                     int64_t* oR, int64_t* oP, plo_orbiter_report* rep) {
  if (!Ln || !Rn || !Pn || !oL || !oR || !oP || !rep || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) {
    plo::set_error("plo_orbiter_modp: bad argument");
    return PLO_E_ARG;
  }
  uint64_t p = q;
  while (p && (p % 2) == 0) p >>= 1;  // :421-422
  if (p == 1) p = 2;
  if (p < 2 || p >= (1ull << 31) || !is_prime(p)) { plo::set_error("plo_orbiter_modp: the modulus (factors of 2 stripped) must be a prime below 2^31"); return PLO_E_ARG; }
  int m, k, n;
  if (const int rc = plo::check_device()) return rc;
  if (const int rc = mm_shape("plo_orbiter_modp", Lcols, Rcols, Prows, &m, &k, &n)) return rc;
  return guarded("plo_orbiter_modp", [&] {
    ZpField Z((int64_t)p);
    const Dense<ZpField> L = load(Z, (size_t)r, (size_t)Lcols, Ln, Ld), R = load(Z, (size_t)r, (size_t)Rcols, Rn, Rd), P = load(Z, (size_t)Prows, (size_t)r, Pn, Pd);
    memset(rep, 0, sizeof(*rep));
    rep->m = m; rep->k = k; rep->n = n;
    auto count = [&](const Dense<ZpField>& M) { for (int64_t e : M.v) if (e != 0) { ++rep->init_nnz; if (!(Z.is_one(e) || Z.is_mone(e))) ++rep->init_nno; } };
    count(L); count(R); count(P);
    rep->init_score = (double)rep->init_nnz;
    std::vector<int32_t> Li(L.v.begin(), L.v.end()), Ri(R.v.begin(), R.v.end()), Pi(P.v.begin(), P.v.end());
    const int rc = plo_orbit_sweep((uint32_t)p, m, k, n, r, Li.data(), Ri.data(), Pi.data(), 1, 1, 1, PLO_MEASURE_NNZ, mode, seed, 0, loops, &rep->best);
    if (rc) return rc;
    const bool improved = orbit_improves(PLO_MEASURE_NNZ, rep->best, rep->init_score, rep->init_nnz, rep->init_nno);
    Dense<ZpField> Lj = L, Rg = R, hP = P;
    if (improved) {
      std::vector<int32_t> U((size_t)m * m), V((size_t)k * k), W((size_t)n * n);
      plo_orbit_decode(m, k, n, mode, seed, rep->best.index, U.data(), V.data(), W.data());
      orbit_transform(Z, m, k, n, r, L, R, P, U, V, W, Lj, Rg, hP);
    }
    rep->improved = improved ? 1 : 0;
    store(Lj, oL, nullptr); store(Rg, oR, nullptr); store(hP, oP, nullptr);
    // MMchecker of the returned triple in the field (:355)
    CsrHost cl, cr, cp;
    to_csr(Lj, cl); to_csr(Rg, cr); to_csr(hP, cp);
    const plo_csr vl = cl.view(r, Lcols), vr = cr.view(r, Rcols), vp = cp.view(Prows, r);
    rep->mm_verdict = plo_mmcheck_batch((uint32_t)p, m, k, n, r, &vl, &vr, &vp, seed ^ 0x4D4D636865636Bull, 32, nullptr, nullptr, nullptr);
    return PLO_OK;
  });
}

int plo_negater(int only_sign, int r, int Lcols, int Rcols, int Prows, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                const int64_t* Pn, const int64_t* Pd, int64_t* oLn, int64_t* oLd, int64_t* oRn, int64_t* oRd, int64_t* oPn, int64_t* oPd,
                uint64_t* stats) {
  if (!Ln || !Rn || !Pn || !oLn || !oLd || !oRn || !oRd || !oPn || !oPd || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) {
    plo::set_error("plo_negater: bad argument");
    return PLO_E_ARG;
  }
  return guarded("plo_negater", [&] {
    QField Q;
    Dense<QField> L = load(Q, (size_t)r, (size_t)Lcols, Ln, Ld), R = load(Q, (size_t)r, (size_t)Rcols, Rn, Rd);
    Dense<QField> Pt = transposed(load(Q, (size_t)Prows, (size_t)r, Pn, Pd));
    const NegaterStats st = Negater().run(L, R, Pt, only_sign != 0);
    store(L, oLn, oLd); store(R, oRn, oRd); store(transposed(Pt), oPn, oPd);
    if (stats) {
      stats[0] = st.gcd_before; stats[1] = st.gcd_after; stats[2] = st.swaps;
      for (int t = 0; t < 3; ++t) { stats[3 + t] = st.neg_before[t]; stats[6 + t] = st.neg_after[t]; stats[9 + t] = st.entries[t]; }
    }
    return PLO_OK;
  });
}

int plo_rotater(int right, int r, int Lcols, int Rcols, int Prows, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                const int64_t* Pn, const int64_t* Pd, int64_t* oLn, int64_t* oLd, int64_t* oRn, int64_t* oRd, int64_t* oPn, int64_t* oPd) {
  if (!Ln || !Rn || !Pn || !oLn || !oLd || !oRn || !oRd || !oPn || !oPd || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) {
    plo::set_error("plo_rotater: bad argument");
    return PLO_E_ARG;
  }
  int m, k, n;
  if (const int rc = mm_shape("plo_rotater", Lcols, Rcols, Prows, &m, &k, &n)) return rc;
  return guarded("plo_rotater", [&] {
    QField Q;
    const Dense<QField> L = load(Q, (size_t)r, (size_t)Lcols, Ln, Ld), R = load(Q, (size_t)r, (size_t)Rcols, Rn, Rd), P = load(Q, (size_t)Prows, (size_t)r, Pn, Pd);
    Dense<QField> Lr, Rr, Pr;
    rotate(right != 0, (size_t)k, (size_t)n, L, R, P, Lr, Rr, Pr);
    store(Lr, oLn, oLd); store(Rr, oRn, oRd); store(Pr, oPn, oPd);
    return PLO_OK;
  });
}

int plo_set_sweep_devices(int n) {
  if (n < 1) { plo::set_error("plo_set_sweep_devices: need n >= 1"); return PLO_E_ARG; }
  g_sweep_devices = n;
  return PLO_OK;
}

// growthfactor  src/growthfactor.cpp:143-231: the growth / error factors of one triple.  G2 (:117-125) is the measure of the orbit
// sweep and comes from the device (plo_growth_G2); the other norms are a few passes over the matrices on the host.
// out[11] = Ginfinf, Ginf2, G2inf, G22, G2, Q0, Qkinfinf, Q1inf2, Q12inf, Qk2inf, Q122   (print order of :199-229)
// q as in load_triple; entry e of a matrix is the double an[e]/ad[e] + bn[e]/bd[e].s (access(), :25-28), s = sqrt(d)
static int growth_factors(int r, int Lcols, int Rcols, int Prows, const int64_t* const q[12], double s, double* out) {
  int m, k, n;
  plo_LRP2MM(Lcols, Rcols, Prows, &m, &k, &n);
  auto dbl = [&](int x, size_t cnt) {
    const int64_t *an = q[4 * x], *ad = q[4 * x + 1], *bn = q[4 * x + 2], *bd = q[4 * x + 3];
    std::vector<double> v(cnt);
    for (size_t e = 0; e < cnt; ++e) {
      const double a = (double)an[e] / (double)(ad ? ad[e] : 1);
      v[e] = bn ? a + (double)bn[e] / (double)(bd ? bd[e] : 1) * s : a;
    }
    return v;
  };
  const std::vector<double> L = dbl(0, (size_t)r * Lcols), R = dbl(1, (size_t)r * Rcols), P = dbl(2, (size_t)Prows * r);
  auto row = [](const std::vector<double>& M, int cols, int i) { return M.data() + (size_t)i * cols; };
  auto norm0 = [](const double* v, int c) { double s = 0; for (int j = 0; j < c; ++j) s += v[j] != 0.0; return s; };             // :32-34
  auto norm1 = [](const double* v, int c) { double s = 0; for (int j = 0; j < c; ++j) s += std::fabs(v[j]); return s; };        // :36-39
  auto norm2 = [](const double* v, int c) { double s = 0; for (int j = 0; j < c; ++j) s += v[j] * v[j]; return std::sqrt(s); };  // :41-44
  std::vector<double> gpinf((size_t)Prows, 0.), gp2((size_t)Prows, 0.);                                                         // :57-67, 87-97
  for (int i = 0; i < r; ++i) {
    const double n1 = norm1(row(L, Lcols, i), Lcols) * norm1(row(R, Rcols, i), Rcols);
    const double n2 = norm2(row(L, Lcols, i), Lcols) * norm2(row(R, Rcols, i), Rcols);
    for (int j = 0; j < Prows; ++j) { const double a = std::fabs(P[(size_t)j * r + i]); gpinf[(size_t)j] += n1 * a; gp2[(size_t)j] += n2 * a; }
  }
  const double ginfinf = *std::max_element(gpinf.begin(), gpinf.end()), ginf2 = *std::max_element(gp2.begin(), gp2.end());
  const double g2inf = norm2(gpinf.data(), Prows), g22 = norm2(gp2.data(), Prows);
  double g2 = 0.;
  const int rc = plo_growth_G2(1, r, Lcols, Rcols, Prows, L.data(), R.data(), P.data(), &g2);
  if (rc) return rc;
  std::vector<double> n0LR((size_t)r);                                                                                          // Q0 :128-143
  for (int i = 0; i < r; ++i) n0LR[(size_t)i] = norm0(row(L, Lcols, i), Lcols) * norm0(row(R, Rcols, i), Rcols);
  double q0 = 0.;
  for (int j = 0; j < Prows; ++j) {
    double rj = 0.;
    for (int i = 0; i < r; ++i) if (P[(size_t)j * r + i] != 0.0 && n0LR[(size_t)i] > rj) rj = n0LR[(size_t)i];
    rj += norm0(row(P, r, j), r);
    if (rj > q0) q0 = rj;
  }
  auto Qk = [](double q, double gamma, double kk) { return q * gamma / std::fabs(gamma - kk); };                                // :145
  const double sqrtk = std::sqrt((double)k), kth = sqrtk * sqrtk * sqrtk;
  const double v[11] = {ginfinf, ginf2, g2inf, g22, g2, q0, Qk(q0, ginfinf, (double)k), Qk(q0, ginf2, 1.), Qk(q0, g2inf, 1.), Qk(q0, g2inf, kth), Qk(q0, g22, 1.)};
  for (int t = 0; t < 11; ++t) out[t] = v[t];
  return PLO_OK;
}

int plo_growth_factors(int r, int Lcols, int Rcols, int Prows, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                       const int64_t* Pn, const int64_t* Pd, double* out) {
  if (!Ln || !Rn || !Pn || !out || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) { plo::set_error("plo_growth_factors: bad argument"); return PLO_E_ARG; }
  const int64_t* const q[12] = {Ln, Ld, nullptr, nullptr, Rn, Rd, nullptr, nullptr, Pn, Pd, nullptr, nullptr};
  return growth_factors(r, Lcols, Rcols, Prows, q, 0., out);
}

// The same factors over Q(sqrt d), d > 0 not a perfect square.
int plo_growth_factors_quad(int64_t d, int r, int Lcols, int Rcols, int Prows, const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn,
                            const int64_t* Lbd, const int64_t* Ran, const int64_t* Rad, const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan,
                            const int64_t* Pad, const int64_t* Pbn, const int64_t* Pbd, double* out) {
  if (!Lan || !Lbn || !Ran || !Rbn || !Pan || !Pbn || !out || r < 1 || Lcols < 1 || Rcols < 1 || Prows < 1) {
    plo::set_error("plo_growth_factors_quad: bad argument");
    return PLO_E_ARG;
  }
  if (const int rc = plo::quad_field_ok(d, PLO_MEASURE_G2, "plo_growth_factors_quad")) return rc;
  const int64_t* const q[12] = {Lan, Lad, Lbn, Lbd, Ran, Rad, Rbn, Rbd, Pan, Pad, Pbn, Pbd};
  return growth_factors(r, Lcols, Rcols, Prows, q, std::sqrt((double)d), out);
}

int plo_mmchecker(uint64_t modulus, uint64_t seed, int batch, int Lrows, int Lcols, int Rrows, int Rcols, int Prows,
                  int Pcols, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                  const int64_t* Pn, const int64_t* Pd, uint32_t* nnz_nno) {
  if (!Ln || !Rn || !Pn || batch < 1 || Lrows < 1 || Lcols < 1 || Rrows < 1 || Rcols < 1 || Prows < 1 || Pcols < 1) {
    plo::set_error("plo_mmchecker: bad argument");
    return PLO_E_ARG;
  }
  const int64_t* const q[12] = {Ln, Ld, nullptr, nullptr, Rn, Rd, nullptr, nullptr, Pn, Pd, nullptr, nullptr};
  return guarded("plo_mmchecker", [&] {
    return mmchecker_triple(load_triple(0, Lrows, Lcols, Rrows, Rcols, Prows, Pcols, q), modulus, 32, seed, batch, nnz_nno, nullptr);
  });
}

int plo_mmchecker_bits(uint64_t modulus, int bitsize, uint64_t seed, int batch, int Lrows, int Lcols, int Rrows, int Rcols, int Prows,
                       int Pcols, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                       const int64_t* Pn, const int64_t* Pd, uint32_t* nnz_nno, int* nprimes) {
  if (!Ln || !Rn || !Pn || batch < 1 || bitsize < 1 || Lrows < 1 || Lcols < 1 || Rrows < 1 || Rcols < 1 || Prows < 1 || Pcols < 1) {
    plo::set_error("plo_mmchecker_bits: bad argument");
    return PLO_E_ARG;
  }
  const int64_t* const q[12] = {Ln, Ld, nullptr, nullptr, Rn, Rd, nullptr, nullptr, Pn, Pd, nullptr, nullptr};
  return guarded("plo_mmchecker_bits", [&] {
    return mmchecker_triple(load_triple(0, Lrows, Lcols, Rrows, Rcols, Prows, Pcols, q), modulus, bitsize, seed, batch, nnz_nno, nprimes);
  });
}

// MMchecker over Q(sqrt d) (`MMchecker -P "X^2-d"`): the exact check of mmcheck_dense at `batch` integer points with `bitsize`-bit
// coordinates, modulo split primes under both embeddings of sqrt(d).
int plo_mmchecker_quad(int64_t d, int bitsize, uint64_t seed, int batch, int Lrows, int Lcols, int Rrows, int Rcols, int Prows, int Pcols,
                       const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn, const int64_t* Lbd, const int64_t* Ran, const int64_t* Rad,
                       const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan, const int64_t* Pad, const int64_t* Pbn, const int64_t* Pbd,
                       uint32_t* nnz_nno, int* nprimes) {
  if (!Lan || !Lbn || !Ran || !Rbn || !Pan || !Pbn || batch < 1 || bitsize < 1 || Lrows < 1 || Lcols < 1 || Rrows < 1 || Rcols < 1 || Prows < 1 ||
      Pcols < 1) {
    plo::set_error("plo_mmchecker_quad: bad argument");
    return PLO_E_ARG;
  }
  if (const int rc = plo::quad_field_ok(d, PLO_MEASURE_NNZ, "plo_mmchecker_quad")) return rc;
  const int64_t* const q[12] = {Lan, Lad, Lbn, Lbd, Ran, Rad, Rbn, Rbd, Pan, Pad, Pbn, Pbd};
  return guarded("plo_mmchecker_quad", [&] {
    return mmchecker_triple(load_triple(d, Lrows, Lcols, Rrows, Rcols, Prows, Pcols, q), 0, bitsize, seed, batch, nnz_nno, nprimes);
  });
}

}  // extern "C"
