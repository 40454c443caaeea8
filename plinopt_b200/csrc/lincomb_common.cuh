// lincomb_common.cuh -- the one design behind both sparsifier search drivers (lincomb_search.cu: one (block,num) step per launch,
// plan API, range sharding, the wide m > 64 path; lincomb_quad.cu: all rows of an inner block in one launch sequence).
//   device core: the packed (rl, cl, -index) key and its decode, the negated prefix sum of a coordinate, the zero count of a T3 row,
//                the block maximum of a key, the field arithmetic and the lazy independence test against annihilator functionals,
//                the inverse-lookup tables and their counting loop;
//   launch:      with_mpad / with_elem (compiled row lengths and element types) and launch (shared-memory attribute);
//   host policy: canonical residues, the exact-path magnitude guard and element width, the inverse-lookup rule, the l-range
//                split, the shared-memory limit, the annihilator functionals of the previous rows.
#pragma once
#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include <utility>
#include <vector>

#include "host/exact.hpp"
#include "plo_device.cuh"

namespace plo {

constexpr int kLcThreads = 128;
constexpr int kIdxBits = 36;
constexpr unsigned long long kIdxMask = (1ull << kIdxBits) - 1ull;
constexpr size_t kSmemLimit = 200 * 1024;  // dynamic shared memory a search kernel may ask for (227 KB per block on a B200)

// key = (rl+1) << 48 | (cl+1) << 36 | (2^36 - 2 - index); the weight seed uses low bits 2^36-1
__host__ __device__ __forceinline__ unsigned long long pack_key(int rl, int cl, unsigned long long low) {
  return ((unsigned long long)(rl + 1) << 48) | ((unsigned long long)(cl + 1) << kIdxBits) | low;
}
inline void unpack_key(unsigned long long key, int& rl, int& cl, uint64_t& index) {
  rl = (int)(key >> 48) - 1;
  cl = (int)((key >> kIdxBits) & 0xFFFull) - 1;
  index = kIdxMask - 1ull - (key & kIdxMask);
}

// ---- device core ------------------------------------------------------------------------------------------------------------------
// prefix q = (i*c + j)*c + k, candidate index = q*c + l
template <typename Q>
__device__ __forceinline__ void decode_prefix(Q q, int c, int& i, int& j, int& k) {
  k = (int)(q % (unsigned)c);
  const Q qq = q / (unsigned)c;
  j = (int)(qq % (unsigned)c);
  i = (int)(qq / (unsigned)c);
}
template <typename Q>
__device__ __forceinline__ void decode_index(Q idx, int c, int& i, int& j, int& k, int& l) {
  l = (int)(idx % (unsigned)c);
  decode_prefix(idx / (unsigned)c, c, i, j, k);
}

// A value no T3 entry takes (residues are below p <= 2^32 - 1, integers below the magnitude bound): padding never counts as a zero.
template <typename T, bool MODP>
__device__ __forceinline__ T pad_sentinel() { return (T)(~(T)0) >> (MODP ? 0 : 1); }
// Coordinate e of nb = -(T0[i][e] + T1[j][e] + T2[.][k]) in the field (past m the caller stores pad_sentinel instead)
template <typename T, bool MODP>
__device__ __forceinline__ T neg_prefix_sum(T a0, T a1, T a2, unsigned int p) {
  if (MODP) {
    unsigned long long sum = (unsigned long long)a0 + a1 + a2;  // < 3p
    sum -= sum >= p ? p : 0u;
    sum -= sum >= p ? p : 0u;
    return (T)(sum ? p - sum : 0ull);
  }
  return (T)0 - (a0 + a1 + a2);
}
// Zero count of one candidate: the coordinates where the T3 row (16-byte aligned, usually shared memory) equals nb.
template <typename T, int LEN>
__device__ __forceinline__ int zero_count(const T* row, const T (&nb)[LEN]) {
  constexpr int VEC = 16 / sizeof(T);  // elements per 128-bit load
  int rl = 0;
#pragma unroll
  for (int e4 = 0; e4 < LEN / VEC; ++e4) {
    const uint4 u = reinterpret_cast<const uint4*>(row)[e4];
    if (sizeof(T) == 4) {
      rl += (nb[e4 * 4 + 0] == (T)u.x);
      rl += (nb[e4 * 4 + 1] == (T)u.y);
      rl += (nb[e4 * 4 + 2] == (T)u.z);
      rl += (nb[e4 * 4 + 3] == (T)u.w);
    } else {
      rl += (nb[e4 * 2 + 0] == (T)(((unsigned long long)u.y << 32) | u.x));
      rl += (nb[e4 * 2 + 1] == (T)(((unsigned long long)u.w << 32) | u.z));
    }
  }
  return rl;
}

// Maximum of v over the THREADS threads of the block; on_thread0(maximum) runs on thread 0.  Every thread calls it with its
// threadIdx.x (read in the kernel, where __launch_bounds__ bounds it) and a 32-word shared buffer; it synchronises the block once.
template <int THREADS, class F>
__device__ __forceinline__ void block_max(unsigned long long v, unsigned tid, unsigned long long* red, F&& on_thread0) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, d);
    v = o > v ? o : v;
  }
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  if (tid < 32) {
    v = tid < (THREADS >> 5) ? red[tid] : 0ull;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, d);
      v = o > v ? o : v;
    }
    if (tid == 0) on_thread0(v);
  }
}

// Field arithmetic of the device: exact in 128 bits, or on canonical residues mod p with Barrett reductions.
template <bool MODP>
struct DevField;
template <>
struct DevField<false> {
  typedef __int128 V;
  unsigned int p;
  __device__ V mul(V a, V b) const { return a * b; }
  __device__ V sub(V a, V b) const { return a - b; }
  __device__ V add(V a, V b) const { return a + b; }
  __device__ V neg(V a) const { return -a; }
  __device__ V from(long long x) const { return (V)x; }
  __device__ V magnitude(V a) const { return a < 0 ? -a : a; }
};
template <>
struct DevField<true> {
  typedef unsigned long long V;
  unsigned int p;
  unsigned long long m64;  // floor((2^64 - 1) / p): Barrett quotient estimate, at most 2 below the true quotient
  __device__ V red(V x) const {
    V r = x - __umul64hi(x, m64) * p;
    r -= r >= p ? p : 0;
    r -= r >= p ? p : 0;
    return r;
  }
  __device__ V mul(V a, V b) const { return red(a * b); }
  __device__ V sub(V a, V b) const { const V r = a + p - b; return r >= p ? r - p : r; }
  __device__ V add(V a, V b) const { const V r = a + b; return r >= p ? r - p : r; }
  __device__ V neg(V a) const { return a ? p - a : 0; }
  __device__ V from(long long x) const { return (V)x; }  // canonical residues in
  __device__ V magnitude(V a) const { return a; }
};

// w = (C_i, C_j, C_k, C_l) is independent of the previous rows iff phi_q . w != 0 for some annihilator functional phi_q.
// Rolled, out of line, Barrett reductions: only a candidate that would beat a running best is tested.
template <bool MODP>
__device__ __noinline__ bool independent(const long long* phi, int nphi, const long long* __restrict__ coef, unsigned int p,
                                         unsigned long long m64, int i, int j, int k, int l) {
  const long long w[4] = {coef[i], coef[j], coef[k], coef[l]};
#pragma unroll 1
  for (int q = 0; q < nphi; ++q) {
    if (MODP) {
      DevField<true> R;
      R.p = p; R.m64 = m64;
      unsigned long long sacc = 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) sacc = R.add(sacc, R.mul((unsigned long long)phi[q * 4 + t], (unsigned long long)w[t]));
      if (sacc) return true;
    } else {
      long long sacc = 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) sacc += phi[q * 4 + t] * w[t];
      if (sacc) return true;
    }
  }
  return false;
}

// ---- launch dispatch ----------------------------------------------------------------------------------------------------------------
// f(std::integral_constant<int, MPAD>) for the compiled row lengths
template <class F>
cudaError_t with_mpad(int mpad, F&& f) {
  switch (mpad) {
    case 8: return f(std::integral_constant<int, 8>{});
    case 16: return f(std::integral_constant<int, 16>{});
    case 32: return f(std::integral_constant<int, 32>{});
    case 48: return f(std::integral_constant<int, 48>{});
    case 64: return f(std::integral_constant<int, 64>{});
    default: return cudaErrorInvalidValue;
  }
}
// f(std::integral_constant<int, WIDTH>, std::integral_constant<bool, MODP>) for the element types: 32-bit residues mod p,
// 32-bit or 64-bit integers
template <int WIDTH>
using elem_t = typename std::conditional<WIDTH == 4, uint32_t, uint64_t>::type;
template <class F>
auto with_elem(uint32_t p, int width, F&& f) {
  if (width == 8) return f(std::integral_constant<int, 8>{}, std::false_type{});
  if (p) return f(std::integral_constant<int, 4>{}, std::true_type{});
  return f(std::integral_constant<int, 4>{}, std::false_type{});
}
// kern<<<grid, threads, smem, st>>>(args...), raising the kernel's dynamic shared-memory limit when it needs more than 48 KB
template <typename... P, typename... A>
cudaError_t launch(void (*kern)(P...), dim3 grid, int threads, size_t smem, cudaStream_t st, A&&... args) {
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<grid, threads, smem, st>>>(std::forward<A>(args)...);
  return cudaGetLastError();
}


// ---- inverse lookup (mod p, many coefficients) ----------------------------------------------------------------------------------
// For a fixed prefix (i,j,k) coordinate e of v vanishes iff  C_l . A3_e = -(s_e),  s_e = C_i A0_e + C_j A1_e + C_k A2_e.  When A3_e is
// invertible that pins the VALUE of C_l: x_e = s_e . (-A3_e^-1); a hash table over the coefficient values turns it into the (usually
// one, possibly zero or several) positions l.  So a prefix costs one multiplication + one probe per coordinate plus a scan of c byte
// counters, instead of c compares per coordinate: ~5x fewer instructions at c = 128 (m = 48).  Exactly the same zero counts.
struct InvTables {           // one problem; lives in global memory, staged into shared memory by each block
  static constexpr unsigned kEmpty = 0xFFFFFFFFu;
  // layout (32-bit words): ninv[mpad] | htab[2 * hsize] (value, first l) | nextdup[c] (next l with the same value, kEmpty: none)
  static __host__ __device__ size_t words(int mpad, int hsize, int c) { return (size_t)mpad + 2 * (size_t)hsize + (size_t)c; }
};
__host__ __device__ __forceinline__ unsigned inv_hash(unsigned x, int hbits) { return (x * 0x9E3779B1u) >> (32 - hbits); }

// ---- host side ----------------------------------------------------------------------------------
inline int pad_m(int m) {
  const int opts[] = {8, 16, 32, 48, 64};
  for (int o : opts) if (m <= o) return o;
  return -1;
}

inline int64_t canonical(uint32_t p, int64_t v) { return p ? (int64_t)(((v % (int64_t)p) + (int64_t)p) % (int64_t)p) : v; }

template <class It>
unsigned __int128 max_abs(It first, It last) {
  unsigned __int128 mx = 0;
  for (; first != last; ++first) {
    const unsigned __int128 a = *first < 0 ? -(__int128)*first : *first;
    if (a > mx) mx = a;
  }
  return mx;
}
// Exact path: a coordinate of v sums four products C.TM, so 4 max|C| max|TM| bounds every table entry and every sum.  Returns the
// element width in bytes (4 when the bound stays below 2^31 - 1), or 0 when the bound reaches 2^62 (the sums would not fit).
inline int exact_width(unsigned __int128 max_coef, unsigned __int128 max_tm) {
  const unsigned __int128 bound = max_coef * max_tm * 4;
  if (bound >= ((unsigned __int128)1 << 62)) return 0;
  return bound < (((unsigned __int128)1 << 31) - 1) ? 4 : 8;
}

// Split the l range of a prefix over lsplit threads until the items of all problems fill every SM four times over, keeping at
// least four l per thread.
inline int lsplit_for(int c, int nproblems, int sms) {
  const unsigned long long nprefix = (unsigned long long)c * c * c;
  const unsigned long long want = (unsigned long long)sms * kLcThreads * 4ull;
  int lsplit = 1;
  while (lsplit < c && nprefix * lsplit * nproblems < want && (c + lsplit * 2 - 1) / (lsplit * 2) >= 4) lsplit *= 2;
  return lsplit;
}

// One reduced functional -> integers: clear denominators over Q; residues are used as they are mod p.
inline void phi_row(const plo::host::QField&, const plo::host::Rat* row, long long* out) {
  // LCD and scaled numerators in 128 bits: a functional that leaves the int64 range throws (PLO_E_RANGE), never wraps
  using plo::host::wide;
  wide lcd = 1;
  for (int t = 0; t < 4; ++t) {
    lcd = lcd / plo::host::wgcd(lcd, row[t].den) * row[t].den;
    if (lcd > (wide)INT64_MAX) throw plo::host::RangeError("annihilator functional: common denominator exceeds 64 bits");
  }
  for (int t = 0; t < 4; ++t) {
    const wide v = (wide)row[t].num * (lcd / row[t].den);
    if (plo::host::wabs(v) > ((wide)1 << 62)) throw plo::host::RangeError("annihilator functional exceeds 62 bits");
    out[t] = (long long)v;
  }
}
inline void phi_row(const plo::host::ZpField&, const int64_t* row, long long* out) {
  for (int t = 0; t < 4; ++t) out[t] = row[t];
}

// Annihilator functionals of span(prev rows) restricted to the live positions off..off+nact-1,
// reduced to an independent set (<= 4 vectors of 4 entries).  Returns false if the previous rows
// are linearly dependent (then rank(Cand) can never exceed num: plinopt_sparsify.inl:173-175).
template <class F>
bool annihilators(const F& f, int n, int nprev, const int64_t* prev, int off, int nact, std::vector<long long>& phi, int& nphi) {
  using namespace plo::host;
  phi.assign(16, 0);
  nphi = 0;
  std::vector<std::vector<typename F::Elt>> basis;
  if (nprev == 0) {
    for (int t = 0; t < nact; ++t) { phi[nphi * 4 + t] = 1; ++nphi; }  // everything non-zero is independent
    return true;
  }
  Dense<F> A(f, (size_t)nprev, (size_t)n);
  for (int i = 0; i < nprev; ++i)
    for (int j = 0; j < n; ++j) A.at(i, j) = f.modular ? f.from_ratio(prev[(size_t)i * n + j], 1) : f.from_int(prev[(size_t)i * n + j]);
  size_t rk = 0;
  basis = nullspace(f, A, &rk);
  if ((int)rk < nprev) return false;
  Dense<F> R(f, basis.size(), 4);
  for (size_t q = 0; q < basis.size(); ++q)
    for (int t = 0; t < nact; ++t) R.at(q, t) = basis[q][off + t];
  const std::vector<size_t> piv = rref(f, R);
  for (size_t q = 0; q < piv.size(); ++q) {
    phi_row(f, &R.at(q, 0), &phi[(size_t)nphi * 4]);
    ++nphi;
  }
  return true;
}


// Builds the inverse-lookup tables of one problem (residues mod an ODD p): a3 = the fourth live row of TM (nullptr / zeros when the block has
// fewer than four live positions), coef = c canonical residues.  ninv[e] = -A3_e^-1 mod p, or kEmpty when A3_e = 0.  The product tables T0, T1,
// T2 of a plan that uses the lookup are PRE-MULTIPLIED by ninv[e] (fold_inv_into_tables on the host, quad_tables_kernel on the device), so
// the value C_l must have at coordinate e is just T0[i][e] + T1[j][e] + T2[e][k] mod p: no multiplication per (prefix, coordinate); the
// kernels read ninv[e] only to tell the coordinates that do not depend on l.  Returns false when some A3_e is not invertible (composite
// modulus).
inline bool build_inv_tables(uint32_t p, int m, int mpad, int c, int hbits, const int64_t* a3, const int64_t* coef, uint32_t* out) {
  const int hsize = 1 << hbits;
  plo::host::ZpField f((int64_t)p);
  uint32_t* ninv = out;
  uint32_t* htab = out + mpad;
  uint32_t* nextdup = htab + 2 * (size_t)hsize;
  for (int e = 0; e < mpad; ++e) {
    const int64_t v = (e < m && a3) ? a3[e] : 0;
    if (v == 0) { ninv[e] = InvTables::kEmpty; continue; }  // the coordinate does not depend on l
    int64_t iv;
    try { iv = f.inv(v); } catch (const plo::host::RangeError&) { return false; }
    ninv[e] = (uint32_t)f.neg(iv);
  }
  for (int h = 0; h < hsize; ++h) { htab[2 * h] = 0; htab[2 * h + 1] = InvTables::kEmpty; }
  for (int l = 0; l < c; ++l) nextdup[l] = InvTables::kEmpty;
  for (int l = c - 1; l >= 0; --l) {  // descending: the head of a chain is its smallest l, chains ascend
    const uint32_t x = (uint32_t)coef[l];
    unsigned h = inv_hash(x, hbits);
    for (;;) {
      if (htab[2 * h + 1] == InvTables::kEmpty) { htab[2 * h] = x; htab[2 * h + 1] = (uint32_t)l; break; }
      if (htab[2 * h] == x) { nextdup[l] = htab[2 * h + 1]; htab[2 * h + 1] = (uint32_t)l; break; }
      h = (h + 1) & (unsigned)(hsize - 1);
    }
  }
  return true;
}
// T0, T1 ([c][mpad]) and T2 ([m][c], transposed) of one problem times ninv[e] where the coordinate depends on l
inline void fold_inv_into_tables(uint32_t p, int m, int mpad, int c, const uint32_t* ninv, uint32_t* t0, uint32_t* t1, uint32_t* t2) {
  for (int e = 0; e < m; ++e) {
    const uint64_t ni = ninv[e];
    if (ni == InvTables::kEmpty) continue;
    for (int l = 0; l < c; ++l) {
      t0[(size_t)l * mpad + e] = (uint32_t)(t0[(size_t)l * mpad + e] * ni % p);
      t1[(size_t)l * mpad + e] = (uint32_t)(t1[(size_t)l * mpad + e] * ni % p);
      t2[(size_t)e * c + l] = (uint32_t)(t2[(size_t)e * c + l] * ni % p);
    }
  }
}
#ifdef __CUDACC__
// The counting loop of the inverse-lookup kernels for ONE prefix (i, j, k): p0 = T0 row i, p1 = T1 row j (m words each), p2 = &T2[0][k]
// (stride c words), all three pre-multiplied by ninv.  Every coordinate costs three loads, two modular additions, one hash probe; a hit increments the byte
// counter of every l with that coefficient value.  Returns the number of coordinates that vanish whatever l is.  The shared-memory
// tables are addressed through 32-bit shared addresses the caller made opaque (under register pressure ptxas re-derives generic
// shared pointers -- S2R + LEA -- inside the loop, ncu profiles/ncu_r02_ad_lincomb_inv_redc.md), the global rows through running
// pointers instead of 64-bit index arithmetic per load.
struct InvShared { uint32_t ninv, htab, nextdup, hist; };  // shared addresses: tables of the problem, byte counters of this thread
__device__ __forceinline__ unsigned inv_count_prefix(const unsigned int* __restrict__ p0, const unsigned int* __restrict__ p1, const unsigned int* __restrict__ p2,
                                                     int c, int m, unsigned int p, int hbits, const InvShared sh) {
  unsigned base = 0;
  const unsigned hmask = (1u << hbits) - 1u;
#pragma unroll 2
  for (int e = 0; e < m; ++e, p2 += c) {
    unsigned int sum = p0[e] + p1[e];  // p <= 2^31: no overflow
    sum -= sum >= p ? p : 0u;
    sum += *p2;
    sum -= sum >= p ? p : 0u;
    unsigned int ni;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(ni) : "r"(sh.ninv + 4u * (unsigned)e));
    if (ni == InvTables::kEmpty) {
      base += (sum == 0u);
    } else {
      const unsigned int x = sum;  // the value C_l must have (the tables carry the factor -A3_e^-1)
      unsigned h = inv_hash(x, hbits);
      for (;;) {
        unsigned int ex, ey;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(ex), "=r"(ey) : "r"(sh.htab + 8u * h));
        if (ey == InvTables::kEmpty) break;
        if (ex == x) {
          for (unsigned l = ey; l != InvTables::kEmpty;) {
            unsigned int v;
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(sh.hist + l));
            asm volatile("st.shared.u8 [%0], %1;" ::"r"(sh.hist + l), "r"(v + 1u) : "memory");
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(l) : "r"(sh.nextdup + 4u * l));
          }
          break;
        }
        h = (h + 1u) & hmask;
      }
    }
  }
  return base;
}
__device__ __forceinline__ InvShared inv_shared_addresses(const void* ninv, const void* htab, const void* nextdup, const void* hist) {
  InvShared s;
  asm volatile("mov.u32 %0, %1;" : "=r"(s.ninv) : "r"((uint32_t)__cvta_generic_to_shared(ninv)));
  asm volatile("mov.u32 %0, %1;" : "=r"(s.htab) : "r"((uint32_t)__cvta_generic_to_shared(htab)));
  asm volatile("mov.u32 %0, %1;" : "=r"(s.nextdup) : "r"((uint32_t)__cvta_generic_to_shared(nextdup)));
  asm volatile("mov.u32 %0, %1;" : "=r"(s.hist) : "r"((uint32_t)__cvta_generic_to_shared(hist)));
  return s;
}
#endif

inline int inv_hash_bits(int c) { int b = 3; while ((1 << b) < 4 * c) ++b; return b; }
// dynamic shared memory of an inverse-lookup count kernel: the problem's tables and c byte counters per thread (rows padded to
// a multiple of 4 plus 4, so that consecutive threads start in different banks)
inline size_t inv_smem_bytes(int mpad, int c) {
  return InvTables::words(mpad, 1 << inv_hash_bits(c), c) * 4 + (size_t)kLcThreads * (((c + 3) & ~3) + 4);
}
// The inverse lookup needs canonical residues mod an odd p <= 2^31 in 32-bit tables (the sum of two residues fits 32 bits)
// and pays off from c = 32 coefficients on.  PLO_LINCOMB_NOINV=1 keeps the compare
// kernels, the reference the lookup is tested against.
inline bool inv_lookup_applies(uint32_t p, int width, int cmin) {
  return p && (p & 1u) && p <= 0x80000000u && width == 4 && cmin >= 32 && getenv("PLO_LINCOMB_NOINV") == nullptr;
}

}  // namespace plo
