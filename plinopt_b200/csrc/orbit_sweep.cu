// orbit_sweep.cu -- DeGroote-orbit candidate sweep on sm_100a.
//
// Replaces the whole candidate loop of the reference's orbiter
//   src/orbiter.cpp:272-324   (omp parallel for + omp critical keep-best)
// One candidate per thread: the (U,V,W) triple is decoded from the candidate
// index (counter-based, DESIGN.md "orbit candidate decode"), the small matrices
// live in registers, the fixed L/R/P (pre-scaled to integers) sit in constant
// memory and are read warp-uniformly, the three Kronecker-product actions
//   L.(U^-1 (x) V), R.(V^-T (x) W), (U (x) W^-1).P        (orbiter.cpp:284-294)
// are evaluated row by row as  U^-T A V,  V^-1 B W,  U C W^-T  without ever
// materialising a Kronecker product, and the measure (nnz/nno: plinopt_library.inl:
// 258-284; G2: growthfactor.cpp:117-125) feeds a warp-shuffle + block argmin.
#include <math.h>
#include <stdlib.h>

#include <cmath>
#include <type_traits>

#include <algorithm>
#include <cstring>
#include <functional>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "plo_device.cuh"

namespace plo {

constexpr int kMaxDim = 8;           // nibble-packed permutations
constexpr int kConstInts = 12000;    // 48 KB of constant memory for L | R | P^T (shipped maximum: 3843 ints, 7686 as int64)
__constant__ __align__(16) int c_lrp[kConstInts];
// Philox round keys of the resident plan's seed (k0 + i.W0, k1 + i.W1, i < 10): loop-invariant, so the table-driven kernels read them
// as constant-bank operands instead of re-deriving them per candidate.
__constant__ uint32_t c_pkeys[20];
constexpr int kConst2Ints = 4300;   // 17 KB: pairs of rows packed at 8-bit spacing for the four-lane kernels
__constant__ __align__(16) int c_lrp2[kConst2Ints];  // int32 entries, or int64 entries (two words each) for the 64-bit input path

#ifndef PLO_SWEEP8_MINB
#define PLO_SWEEP8_MINB 3
#endif
#ifndef PLO_SWEEPN8_MINB
#define PLO_SWEEPN8_MINB 4
#endif
constexpr int MEASURE_BOTH = 4;

// Survivor compaction inside the sweep kernels (north_star: "surviving candidates are compacted through coalesced vectorised
// stores"; reference analogue: the per-improvement report of src/orbiter.cpp:300-318).  While a survivors call runs, the constant
// bank holds a threshold on the sweep's own key and an index buffer: every kernel of the family appends the index of a candidate
// whose key does not exceed the threshold (warp-aggregated: one atomicAdd per warp with survivors, consecutive 8-byte slots).
// idx == nullptr (the normal state) disables it at the cost of one uniform compare per candidate.
struct Surv {
  unsigned long long thr;
  unsigned long long* idx;
  unsigned long long* count;
  unsigned long long cap;
};
__constant__ Surv c_surv;  // internal: nnz, nno and G2 (tables, winner re-evaluation)

// ---------------------------------------------------------------------------
// Digit stream: a pure function of (mode, seed, index).
//   mode 0: digits are the mixed-radix expansion of index (least significant first)
//   mode 1: words w_t = Philox4x32-10(key = seed, counter = (index, t/4))[t%4];
//           a digit of radix rho is taken from the current word x by
//           d = (x*rho) >> 32, x = (x*rho) mod 2^32; a fresh word is fetched at
//           the start of every matrix and whenever the product of the radices
//           taken from the current word would exceed 2^20.
// All bookkeeping (R, nwords) is compile-time constant once the loops are unrolled.
// ---------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ void philox4x32_10_ck(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ c_pkeys[2 * r], n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ c_pkeys[2 * r + 1], n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
#endif

template <int MODE, bool CK = false>
struct Digits {
  unsigned long long index, seed, rem;
  uint32_t x, R, nwords;
  uint32_t buf[4];
  __host__ __device__ __forceinline__ Digits(unsigned long long seed_, unsigned long long index_)
      : index(index_), seed(seed_), rem(index_), x(0), R(0), nwords(0) {}
  __host__ __device__ __forceinline__ void new_word() {
    if ((nwords & 3u) == 0) {
#ifdef __CUDA_ARCH__
      if (CK) philox4x32_10_ck((uint32_t)index, (uint32_t)(index >> 32), nwords >> 2, 0u, buf);
      else
#endif
        philox4x32_10((uint32_t)index, (uint32_t)(index >> 32), nwords >> 2, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), buf);
    }
    x = buf[nwords & 3u];
    ++nwords;
    R = 1;
  }
  __host__ __device__ __forceinline__ void start_matrix() {
    if (MODE == 1) new_word();
  }
  __host__ __device__ __forceinline__ uint32_t digit(uint32_t radix) {
    if (MODE == 0) {
      const uint32_t d = (uint32_t)(rem % radix);
      rem /= radix;
      return d;
    }
    if (R * radix > (1u << 20)) new_word();
    const unsigned long long t = (unsigned long long)x * radix;
    x = (uint32_t)t;
    R *= radix;
    return (uint32_t)(t >> 32);
  }
  // All digits of one matrix at once, when the product `count` of its radices is small: successive multiply-high digits of one word
  // are the mixed-radix digits (first drawn = most significant) of floor(x * count / 2^32); in mode 0 they are those of rem % count
  // (first drawn = least significant).  RawDigits replays either numbering.
  __host__ __device__ __forceinline__ uint32_t matrix_index(uint32_t count) {
    if (MODE == 0) {
      const uint32_t d = (uint32_t)(rem % count);
      rem /= count;
      return d;
    }
    new_word();
#ifdef __CUDA_ARCH__
    return __umulhi(x, count);
#else
    return (uint32_t)(((unsigned long long)x * count) >> 32);
#endif
  }
};

// Digit source that replays matrix number e of `count` (see Digits::matrix_index); no Philox behind it.
template <int MODE>
struct RawDigits {
  unsigned long long rem;
  uint32_t x;
  __host__ __device__ __forceinline__ RawDigits(uint32_t e, uint32_t count)
      : rem(e), x((uint32_t)((((unsigned long long)e << 32) + count - 1) / count)) {}
  __host__ __device__ __forceinline__ void start_matrix() {}
  __host__ __device__ __forceinline__ uint32_t digit(uint32_t radix) {
    if (MODE == 0) {
      const uint32_t d = (uint32_t)(rem % radix);
      rem /= radix;
      return d;
    }
    const unsigned long long t = (unsigned long long)x * radix;
    x = (uint32_t)t;
    return (uint32_t)(t >> 32);
  }
};

// Compact form of one zoi matrix  M[P[i]][Q[j]] = T[i][j]  (src/orbiter.cpp:125-136):
// nibble-packed permutations, sign bits of the diagonal, 2-bit trits of the
// strict upper triangle (row-major over i<j, stored as value+1).
struct Zoi {
  uint32_t pP, pQ, D;
  unsigned long long T;
};

__host__ __device__ __forceinline__ uint32_t nibble_swap(uint32_t perm, int i, uint32_t d) {
  // swap entries i and i+d of a nibble-packed permutation (Fisher-Yates step)
  const uint32_t sh = 4u * (uint32_t)i, sh2 = sh + 4u * d;
  const uint32_t xr = ((perm >> sh) ^ (perm >> sh2)) & 15u;
  return perm ^ (xr << sh) ^ (xr << sh2);
}

template <int S, int MODE, class DS = Digits<MODE>>
__host__ __device__ __forceinline__ Zoi decode_zoi(DS& ds) {
  Zoi z;
  ds.start_matrix();
  z.pP = 0x76543210u;
  z.pQ = 0x76543210u;
#pragma unroll
  for (int i = 0; i + 1 < S; ++i) z.pP = nibble_swap(z.pP, i, ds.digit((uint32_t)(S - i)));
#pragma unroll
  for (int i = 0; i + 1 < S; ++i) z.pQ = nibble_swap(z.pQ, i, ds.digit((uint32_t)(S - i)));
  z.D = 0;
#pragma unroll
  for (int i = 0; i < S; ++i) z.D |= ds.digit(2u) << i;
  z.T = 0;
  int idx = 0;
#pragma unroll
  for (int i = 0; i < S; ++i)
#pragma unroll
    for (int j = i + 1; j < S; ++j) {
      z.T |= (unsigned long long)ds.digit(3u) << (2 * idx);
      ++idx;
    }
  return z;
}

// Classes of a 2x2 zoi matrix M = Pi_P T Pi_Q^T, T = [d0 t; 0 d1].  Permutations and signs on the outer side of a factor change no
// Frobenius norm, zero count or +-1 count, and T = diag(d0, d1).[1 d0.t; 0 1] = [1 t.d1; 0 1].diag(d0, d1), so
//   as a left factor (U^-T.A, U.C) M acts on every measure of its product only through cl(M) = (Q[0], t.d0),
//   as a right factor (A.V, V^-1.B, C.W^-T) only through cr(M) = (P[0], t.d1).
// Both are encoded 3 . bit + (coefficient + 1), in [0, 6).
constexpr int kZ2Classes = 6;
__host__ __device__ __forceinline__ int zoi2_cl(const Zoi& z) {
  return 3 * (int)((z.pQ & 15u) != 0u) + 1 + ((int)(z.T & 3ull) - 1) * ((z.D & 1u) ? 1 : -1);
}
__host__ __device__ __forceinline__ int zoi2_cr(const Zoi& z) {
  return 3 * (int)((z.pP & 15u) != 0u) + 1 + ((int)(z.T & 3ull) - 1) * ((z.D & 2u) ? 1 : -1);
}

// Expand a Zoi into the dense matrix (INV = false) or its inverse (INV = true),
// row-major in out[S*S].  `scr` is a thread-private scratch of S*S ints with
// element stride `stride` (shared memory on the device: out-of-order writes at
// data-dependent positions, then an in-order read back into registers).
//   M     = Pi_P . T . Pi_Q^T      =>  M[P[i]][Q[j]]      = T[i][j]
//   M^-1  = Pi_Q . T^-1 . Pi_P^T   =>  M^-1[Q[i]][P[j]]   = T^-1[i][j]
// T is upper triangular with +-1 diagonal, so T^-1 is integral
// (reference: inverse / inverseTranspose, plinopt_sparsify.inl:380-465).
template <int S, bool INV>
__host__ __device__ __forceinline__ void expand_zoi(const Zoi& z, int* out, volatile int* scr, int stride) {
  if (S == 1) {
    out[0] = (z.D & 1u) ? 1 : -1;
    return;
  }
  if (S == 2) {
    // T = [d0 t; 0 d1], T^-1 = [d0 -d0 t d1; 0 d1]; a 2x2 permutation is identity or swap, so
    // M[a][b] = T[a^sp][b^sq] and M^-1[a][b] = T^-1[a^sq][b^sp]: four selects, no scratch.
    const int d0 = (z.D & 1u) ? 1 : -1, d1 = (z.D & 2u) ? 1 : -1;
    const int tt = (int)(z.T & 3ull) - 1;
    const int off = INV ? -d0 * tt * d1 : tt;
    const bool sp = (z.pP & 15u) != 0u, sq = (z.pQ & 15u) != 0u;
    const bool sr = INV ? sq : sp, sc = INV ? sp : sq;  // row / column swaps
    // rows of T (or T^-1): r0 = (d0, off), r1 = (0, d1)
    const int a0 = sr ? 0 : d0, a1 = sr ? d1 : off;   // row 0 before the column swap
    const int b0 = sr ? d0 : 0, b1 = sr ? off : d1;   // row 1 before the column swap
    out[0] = sc ? a1 : a0; out[1] = sc ? a0 : a1;
    out[2] = sc ? b1 : b0; out[3] = sc ? b0 : b1;
    return;
  }
  int t[S][S];
  {
    int idx = 0;
#pragma unroll
    for (int i = 0; i < S; ++i) {
      t[i][i] = ((z.D >> i) & 1u) ? 1 : -1;
#pragma unroll
      for (int j = i + 1; j < S; ++j) {
        t[i][j] = (int)((z.T >> (2 * idx)) & 3ull) - 1;
        ++idx;
      }
    }
  }
  if (INV) {
    // back substitution: x[i][i] = d_i ; x[i][j] = -d_i * sum_{k=i+1..j} t[i][k] x[k][j]
    int xinv[S][S];
#pragma unroll
    for (int j = 0; j < S; ++j) {
      xinv[j][j] = t[j][j];
#pragma unroll
      for (int i = j - 1; i >= 0; --i) {
        int s = 0;
#pragma unroll
        for (int k = i + 1; k <= j; ++k) s += t[i][k] * xinv[k][j];
        xinv[i][j] = -t[i][i] * s;
      }
    }
#pragma unroll
    for (int i = 0; i < S; ++i)
#pragma unroll
      for (int j = i; j < S; ++j) t[i][j] = xinv[i][j];
  }
#pragma unroll
  for (int e = 0; e < S * S; ++e) scr[e * stride] = 0;
#pragma unroll
  for (int i = 0; i < S; ++i) {
#pragma unroll
    for (int j = i; j < S; ++j) {
      const int Pi = (int)((z.pP >> (4 * (INV ? j : i))) & 15u);
      const int Qj = (int)((z.pQ >> (4 * (INV ? i : j))) & 15u);
      const int pos = INV ? (Qj * S + Pi) : (Pi * S + Qj);
      scr[pos * stride] = t[i][j];
    }
  }
#pragma unroll
  for (int e = 0; e < S * S; ++e) out[e] = scr[e * stride];
}

// ---------------------------------------------------------------------------
// Triangular right factors.  A zoi matrix is M = Pi_P T Pi_Q^T with T upper triangular, diagonal d_i = +-1 (src/orbiter.cpp:
// 125-136).  As the RIGHT factor of a product X.M (or X.M^-T) the outer permutation Pi_Q and the diagonal signs only permute the
// output entries and flip their signs -- every measure (zero count, +-1 count, sum of squares) is blind to both -- and the inner
// permutation Pi_P permutes the entries of X:
//     (X.M)[Q[j]]    = d_j  ( X'[j] + sum_{i<j} X'[i] . T[i][j] d_j )           X'[i] = X[P[i]]
//     (X.M^-T)[Q[i]] = d_i  ( X'[i] + sum_{j>i} X'[j] . d_i T^-1[i][j] )
// so the second product stage costs S(S-1)/2 multiply-adds per row of X instead of S^2 (7x7: 21 instead of 49), the unit diagonal
// is the accumulator's start value, and the factor occupies S(S-1)/2 registers instead of S^2.  X is permuted through the
// thread-private column of the expansion scratch (S stores, S loads, bank-conflict free).
// tri[i*S - i(i+1)/2 + (j-i-1)] for i < j:   INV = false: T[i][j].d_j     INV = true: d_i.T^-1[i][j]
// ---------------------------------------------------------------------------
template <int S>
__host__ __device__ constexpr int tri_index(int i, int j) { return i * S - i * (i + 1) / 2 + (j - i - 1); }

template <int S, bool INV>
__host__ __device__ __forceinline__ void zoi_tri(const Zoi& z, int* tri) {
  int t[S][S];
  {
    int idx = 0;
#pragma unroll
    for (int i = 0; i < S; ++i) {
      t[i][i] = ((z.D >> i) & 1u) ? 1 : -1;
#pragma unroll
      for (int j = i + 1; j < S; ++j) {
        t[i][j] = (int)((z.T >> (2 * idx)) & 3ull) - 1;
        ++idx;
      }
    }
  }
  if (!INV) {
#pragma unroll
    for (int i = 0; i < S; ++i)
#pragma unroll
      for (int j = i + 1; j < S; ++j) tri[tri_index<S>(i, j)] = t[i][j] * t[j][j];
  } else {
    int xinv[S][S];  // back substitution, as in expand_zoi
#pragma unroll
    for (int j = 0; j < S; ++j) {
      xinv[j][j] = t[j][j];
#pragma unroll
      for (int i = j - 1; i >= 0; --i) {
        int acc = 0;
#pragma unroll
        for (int k = i + 1; k <= j; ++k) acc += t[i][k] * xinv[k][j];
        xinv[i][j] = -t[i][i] * acc;
      }
    }
#pragma unroll
    for (int i = 0; i < S; ++i)
#pragma unroll
      for (int j = i + 1; j < S; ++j) tri[tri_index<S>(i, j)] = t[i][i] * xinv[i][j];
  }
}
// scratch offsets (in ints, thread-private column with stride kThreads) of X[P[i]]
template <int S>
__device__ __forceinline__ void zoi_perm_offsets(const Zoi& z, int stride, int* poff) {
#pragma unroll
  for (int i = 0; i < S; ++i) poff[i] = (int)((z.pP >> (4 * i)) & 15u) * stride;
}

// ---------------------------------------------------------------------------
// Per-row scoring.  Y = Lm' . A . Rm'  with A (RA x CA) read warp-uniformly,
// Lm' = Lm or Lm^T, Rm' = Rm or Rm^T; every entry of Y goes to the accumulator.
// ---------------------------------------------------------------------------
struct Acc {
  int nnz, nno, sq;
};

// `den` is the common denominator of the matrix: the true entry is y/den, so it is +-1 iff |y| == den
// (isAbsOne, include/plinopt_library.h:188-191).
template <int MEASURE>
__host__ __device__ __forceinline__ void consume(Acc& a, int y, int den) {
  if (MEASURE == PLO_MEASURE_NNZ || MEASURE == MEASURE_BOTH) {
    a.nnz += (y != 0);
    a.nno += (y != 0) & (y != den) & (y != -den);
  }
  if (MEASURE == PLO_MEASURE_G2 || MEASURE == MEASURE_BOTH) a.sq += y * y;
}

template <int RA, int CA, bool TL, bool TR, int MEASURE>
__host__ __device__ __forceinline__ void transform_row(const int* __restrict__ A, const int* Lm, const int* Rm, int den, Acc& acc) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A[e];
#pragma unroll
  for (int x = 0; x < RA; ++x) {
    int X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      int s = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) s += (TL ? Lm[i * RA + x] : Lm[x * RA + i]) * a[i * CA + j];
      X[j] = s;
    }
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      int s = 0;
#pragma unroll
      for (int j = 0; j < CA; ++j) s += X[j] * (TR ? Rm[y * CA + j] : Rm[j * CA + y]);
      consume<MEASURE>(acc, s, den);
    }
  }
}

// ---------------------------------------------------------------------------
// Two-lane variant: two rows x0,x1 of Y = Lm'.A.Rm' travel in one 32-bit register as
// v = y[x0] + 65536*y[x1] (plain integer arithmetic is linear in this encoding, so both stages
// of the product act on both lanes with ONE IMAD each); lanes are split only to be scored:
// hi = (v + 0x8000) >> 16, lo = sign-extended low half.  Valid while every |entry| < 2^15
// (host-side magnitude bound).  Halves the IMAD count of the transforms.
// ---------------------------------------------------------------------------
template <int RA, bool TL>
__device__ __forceinline__ void pack_left(const int* Lm, int* LmP) {
  // LmP[xp*RA + i] = Lm'[2xp][i] + (Lm'[2xp+1][i] << 16), Lm' = TL ? Lm^T : Lm
#pragma unroll
  for (int xp = 0; xp < (RA + 1) / 2; ++xp)
#pragma unroll
    for (int i = 0; i < RA; ++i) {
      const int x0 = 2 * xp, x1 = 2 * xp + 1;
      const int lo = TL ? Lm[i * RA + x0] : Lm[x0 * RA + i];
      const int hi = x1 < RA ? (TL ? Lm[i * RA + x1] : Lm[x1 * RA + i]) : 0;
      LmP[xp * RA + i] = lo + hi * 65536;
    }
}


// ---------------------------------------------------------------------------
// 2x2 zoi matrices: the group has 2.2.2.2.3 = 48 elements, so decode + expansion + inverse + lane packing become one table in
// shared memory, built by each block with the generic code above (same digits -> same matrices) and indexed by
// Digits::matrix_index(48).  Entry layout (kZ2Stride = 20 words = 80 B: eight consecutive entries start in eight different
// 16-byte bank groups):  M (4) | M^-1 (4) | pack_left<T>(M^-1) (2) | pack_left(M) (2) | pack_left(M^-1) (2).
// ---------------------------------------------------------------------------
constexpr int kZ2Count = 48, kZ2Stride = 20;
#ifdef __CUDACC__
template <int MODE>
__device__ __forceinline__ void build_zoi2_table(int* tab) {
  for (int e = threadIdx.x; e < kZ2Count; e += blockDim.x) {
    RawDigits<MODE> ds((uint32_t)e, (uint32_t)kZ2Count);
    const Zoi z = decode_zoi<2, MODE, RawDigits<MODE>>(ds);
    int Mx[4], Mi[4], pit[2], pm[2], pi[2];
    expand_zoi<2, false>(z, Mx, nullptr, 0);
    expand_zoi<2, true>(z, Mi, nullptr, 0);
    pack_left<2, true>(Mi, pit);
    pack_left<2, false>(Mx, pm);
    pack_left<2, false>(Mi, pi);
    int* t = tab + e * kZ2Stride;
#pragma unroll
    for (int q = 0; q < 4; ++q) { t[q] = Mx[q]; t[4 + q] = Mi[q]; }
    t[8] = pit[0]; t[9] = pit[1]; t[10] = pm[0]; t[11] = pm[1]; t[12] = pi[0]; t[13] = pi[1];
  }
}
__device__ __forceinline__ void z2_load4(const int* t, int* out) {
  const int4 v = *reinterpret_cast<const int4*>(t);
  out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
}
__device__ __forceinline__ void z2_load2(const int* t, int* out) {
  const int2 v = *reinterpret_cast<const int2*>(t);
  out[0] = v.x; out[1] = v.y;
}
#endif

template <int RA, int CA, bool TR, int MEASURE>
__device__ __forceinline__ void transform_row_packed(const int* __restrict__ A, const int* LmP, const int* Rm, int den, Acc& acc) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A[e];
#pragma unroll
  for (int xp = 0; xp < (RA + 1) / 2; ++xp) {
    int X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      int s = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) s += LmP[xp * RA + i] * a[i * CA + j];
      X[j] = s;
    }
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      int v = 0;
#pragma unroll
      for (int j = 0; j < CA; ++j) v += X[j] * (TR ? Rm[y * CA + j] : Rm[j * CA + y]);
      if (MEASURE == PLO_MEASURE_NNZ) {
        // both lanes are classified in packed form (DPX 16x2 min): w holds lane + 0x8000 in each half (the +0x8000 of the low
        // half also absorbs the borrow of the encoding), a half of w ^ c is zero iff the lane equals c - 0x8000.
        // acc.nnz += [lane != 0], acc.nno += [|lane| != den], per half; score_candidate turns the second count into nno
        // (a phantom upper lane of an odd last pair is 0: it adds nothing to nnz and 1 to the second count, like every zero).
        const unsigned w = (unsigned)v + 0x80008000u;
        const unsigned d2 = (unsigned)den * 0x00010001u;
        // a run-time spelling of 0x00010001 (den > 0): ptxas keeps it in ONE register instead of rematerialising an immediate
        // for every value (the instruction takes a single immediate)
        const unsigned k1 = 0x00010001u + ((unsigned)den >> 31);
        acc.nnz += (int)__viaddmin_u16x2(w, 0x80008000u, k1);  // per-half (w + 0x8000) mod 2^16 = the lane itself; min(lane, 1)
        acc.nno += (int)__vimin3_u16x2(w ^ (0x80008000u + d2), w ^ (0x80008000u - d2), 0x00010001u);
      } else {
        const int hi = (v + 0x8000) >> 16;
        const int lo = (int)(short)(v & 0xFFFF);
        consume<MEASURE>(acc, lo, den);
        if (2 * xp + 1 < RA) consume<MEASURE>(acc, hi, den);
      }
    }
  }
}

struct Score {
  uint32_t nnz, nno;
  double g2;
};

// Scores one candidate.  lrp = L (r x MK) | R (r x KN) | P^T (r x MN), ints.
// sqrt of a small non-negative integer: table lookup (the table holds the correctly rounded
// sqrt((double)s), so the value is bit-identical to computing it).  LF = the table covers every
// reachable value (host-side bound); otherwise values beyond the table take an out-of-line sqrt.
#ifdef __CUDACC__
__device__ __noinline__ double slow_isqrt(int s) { return sqrt((double)s); }
#endif
template <bool LF>
__host__ __device__ __forceinline__ double isqrt_lut(int s, const double* lut, int lutn) {
#ifdef __CUDA_ARCH__
  if (LF || s < lutn) return lut[s];
  return slow_isqrt(s);
#else
  (void)lut; (void)lutn;
  return std::sqrt((double)s);
#endif
}

template <int M, int K, int N, int MODE, int MEASURE, int RU = 0, bool LF = false, bool PACK = false, bool TAB = false>
__host__ __device__ __forceinline__ Score score_candidate(const int* __restrict__ lrp, int r, int3 den, unsigned long long seed,
                                                          unsigned long long index, volatile int* scr, int stride,
                                                          const double* lut = nullptr, int lutn = 0, const int* z2tab = nullptr) {
  static_assert(!TAB || (PACK && M == 2 && K == 2 && N == 2), "table path: packed 2x2x2 only");
  Digits<MODE> ds(seed, index);
  int U[M * M], Ui[M * M], V[K * K], Vi[K * K], W[N * N], Wi[N * N];
#ifdef __CUDA_ARCH__
  int UiTP[((M + 1) / 2) * M], ViP[((K + 1) / 2) * K], UP[((M + 1) / 2) * M];
  if (TAB) {  // 2x2x2 with lane packing: everything the transforms need comes out of the 48-entry table
    const int* tu = z2tab + ds.matrix_index(kZ2Count) * kZ2Stride;
    const int* tv = z2tab + ds.matrix_index(kZ2Count) * kZ2Stride;
    const int* tw = z2tab + ds.matrix_index(kZ2Count) * kZ2Stride;
    int both[4];
    z2_load4(tu + 8, both);
    UiTP[0] = both[0]; UiTP[1] = both[1]; UP[0] = both[2]; UP[1] = both[3];
    z2_load4(tv, V);
    z2_load2(tv + 12, ViP);
    z2_load4(tw, W);
    z2_load4(tw + 4, Wi);
  } else
#endif
  {
    const Zoi zu = decode_zoi<M, MODE>(ds);
    const Zoi zv = decode_zoi<K, MODE>(ds);
    const Zoi zw = decode_zoi<N, MODE>(ds);
    expand_zoi<M, false>(zu, U, scr, stride);
    expand_zoi<M, true>(zu, Ui, scr, stride);
    expand_zoi<K, false>(zv, V, scr, stride);
    expand_zoi<K, true>(zv, Vi, scr, stride);
    expand_zoi<N, false>(zw, W, scr, stride);
    expand_zoi<N, true>(zw, Wi, scr, stride);
#ifdef __CUDA_ARCH__
    if (PACK) {
      pack_left<M, true>(Ui, UiTP);
      pack_left<K, false>(Vi, ViP);
      pack_left<M, false>(U, UP);
    }
#endif
  }

  const int* Lc = lrp;
  const int* Rc = lrp + r * M * K;
  const int* Pc = Rc + r * K * N;
  Score sc;
  sc.nnz = 0; sc.nno = 0; sc.g2 = 0.0;
  int nnz = 0, nno = 0;
  const int rows = RU > 0 ? RU : r;
#ifdef __CUDA_ARCH__
  if (PACK && MEASURE == PLO_MEASURE_NNZ) {
    // packed per-half counters run over ALL rows (rows . lanes < 2^16) and are split once:
    // nnz = sum of halves; nno = nnz - #(|y| == den) = nnz - (lanes - #(|y| != den))
    Acc aL, aR, aP;
    aL.nnz = aL.nno = aL.sq = 0;
    aR = aL; aP = aL;
#pragma unroll(RU > 0 ? RU : 1)
    for (int l = 0; l < rows; ++l) {
      transform_row_packed<M, K, false, MEASURE>(Lc + l * M * K, UiTP, V, den.x, aL);
      transform_row_packed<K, N, false, MEASURE>(Rc + l * K * N, ViP, W, den.y, aR);
      transform_row_packed<M, N, true, MEASURE>(Pc + l * M * N, UP, Wi, den.z, aP);
    }
    constexpr int lanes = 2 * ((M + 1) / 2) * K + 2 * ((K + 1) / 2) * N + 2 * ((M + 1) / 2) * N;
    const int z = (aL.nnz & 0xFFFF) + (aL.nnz >> 16) + (aR.nnz & 0xFFFF) + (aR.nnz >> 16) + (aP.nnz & 0xFFFF) + (aP.nnz >> 16);
    const int d = (aL.nno & 0xFFFF) + (aL.nno >> 16) + (aR.nno & 0xFFFF) + (aR.nno >> 16) + (aP.nno & 0xFFFF) + (aP.nno >> 16);
    sc.nnz = (uint32_t)z;
    sc.nno = (uint32_t)(z - (rows * lanes - d));
    return sc;
  }
#endif
#pragma unroll(RU > 0 ? RU : 1)
  for (int l = 0; l < rows; ++l) {
    Acc aL, aR, aP;
    aL.nnz = aL.nno = aL.sq = 0;
    aR = aL; aP = aL;
#ifdef __CUDA_ARCH__
    if (PACK) {
      transform_row_packed<M, K, false, MEASURE>(Lc + l * M * K, UiTP, V, den.x, aL);
      transform_row_packed<K, N, false, MEASURE>(Rc + l * K * N, ViP, W, den.y, aR);
      transform_row_packed<M, N, true, MEASURE>(Pc + l * M * N, UP, Wi, den.z, aP);
    } else
#endif
    {
      transform_row<M, K, true, false, MEASURE>(Lc + l * M * K, Ui, V, den.x, aL);   // U^-T A V
      transform_row<K, N, false, false, MEASURE>(Rc + l * K * N, Vi, W, den.y, aR);  // V^-1 B W
      transform_row<M, N, false, true, MEASURE>(Pc + l * M * N, U, Wi, den.z, aP);   // U C W^-T
    }
    nnz += aL.nnz + aR.nnz + aP.nnz;
    nno += aL.nno + aR.nno + aP.nno;
    if (MEASURE == PLO_MEASURE_G2 || MEASURE == MEASURE_BOTH) {
      // growthfactor.cpp:117-125: s += norm2(L[i])*norm2(R[i])*norm2(Pt[i]); no FMA contraction
#ifdef __CUDA_ARCH__
      const double t = __dmul_rn(__dmul_rn(isqrt_lut<LF>(aL.sq, lut, lutn), isqrt_lut<LF>(aR.sq, lut, lutn)), isqrt_lut<LF>(aP.sq, lut, lutn));
      sc.g2 = __dadd_rn(sc.g2, t);
#else
      const double t = (std::sqrt((double)aL.sq) * std::sqrt((double)aR.sq)) * std::sqrt((double)aP.sq);
      sc.g2 = sc.g2 + t;
#endif
    }
  }
  sc.nnz = (uint32_t)nnz;
  sc.nno = (uint32_t)nno;
  return sc;
}

// Sparsity score of one candidate in three phases (all rows of L, then of R, then of P): the counts are sums over the three products, so
// only the matrices of ONE product are live at a time -- U^-T and V, then V^-1 and W, then U and W^-T -- instead of all six (3x4x7:
// 134 registers of matrices).  The packed per-half counters run over all rows of a phase (r . lanes < 2^16, checked on the host).
#ifdef __CUDACC__
template <int M, int K, int N, int MODE>
__device__ __forceinline__ Score score_candidate_nnz_split(const int* __restrict__ lrp, int r, int3 den, unsigned long long seed,
                                                           unsigned long long index, volatile int* scr, int stride) {
  Digits<MODE> ds(seed, index);
  const Zoi zu = decode_zoi<M, MODE>(ds);
  const Zoi zv = decode_zoi<K, MODE>(ds);
  const Zoi zw = decode_zoi<N, MODE>(ds);
  const int* Lc = lrp;
  const int* Rc = lrp + r * M * K;
  const int* Pc = Rc + r * K * N;
  Acc aL, aR, aP;
  aL.nnz = aL.nno = aL.sq = 0;
  aR = aL; aP = aL;
  {
    int Ui[M * M], V[K * K], UiTP[((M + 1) / 2) * M];
    expand_zoi<M, true>(zu, Ui, scr, stride);
    pack_left<M, true>(Ui, UiTP);
    expand_zoi<K, false>(zv, V, scr, stride);
#pragma unroll 2
    for (int l = 0; l < r; ++l) transform_row_packed<M, K, false, PLO_MEASURE_NNZ>(Lc + l * M * K, UiTP, V, den.x, aL);   // U^-T A V
  }
  {
    int Vi[K * K], W[N * N], ViP[((K + 1) / 2) * K];
    expand_zoi<K, true>(zv, Vi, scr, stride);
    pack_left<K, false>(Vi, ViP);
    expand_zoi<N, false>(zw, W, scr, stride);
#pragma unroll 2
    for (int l = 0; l < r; ++l) transform_row_packed<K, N, false, PLO_MEASURE_NNZ>(Rc + l * K * N, ViP, W, den.y, aR);    // V^-1 B W
  }
  {
    int U[M * M], Wi[N * N], UP[((M + 1) / 2) * M];
    expand_zoi<M, false>(zu, U, scr, stride);
    pack_left<M, false>(U, UP);
    expand_zoi<N, true>(zw, Wi, scr, stride);
#pragma unroll 2
    for (int l = 0; l < r; ++l) transform_row_packed<M, N, true, PLO_MEASURE_NNZ>(Pc + l * M * N, UP, Wi, den.z, aP);     // U C W^-T
  }
  constexpr int lanes = 2 * ((M + 1) / 2) * K + 2 * ((K + 1) / 2) * N + 2 * ((M + 1) / 2) * N;
  const int z = (aL.nnz & 0xFFFF) + (aL.nnz >> 16) + (aR.nnz & 0xFFFF) + (aR.nnz >> 16) + (aP.nnz & 0xFFFF) + (aP.nnz >> 16);
  const int d = (aL.nno & 0xFFFF) + (aL.nno >> 16) + (aR.nno & 0xFFFF) + (aR.nno >> 16) + (aP.nno & 0xFFFF) + (aP.nno >> 16);
  Score sc;
  sc.nnz = (uint32_t)z;
  sc.nno = (uint32_t)(z - (r * lanes - d));
  sc.g2 = 0.0;
  return sc;
}
#endif

#ifdef __CUDACC__
__device__ __forceinline__ void surv_emit(const Key& k) {
  if (c_surv.idx != nullptr && k.primary <= c_surv.thr) {
    const unsigned act = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs(act) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(c_surv.count, (unsigned long long)__popc(act));
    base = __shfl_sync(act, base, leader);
    const unsigned long long pos = base + __popc(act & ((1u << lane) - 1u));
    if (pos < c_surv.cap) c_surv.idx[pos] = k.index;
  }
}
#endif

template <int MEASURE>
__device__ __forceinline__ Key make_key(const Score& s, unsigned long long index) {
  Key k;
  if (MEASURE == PLO_MEASURE_NNZ) k.primary = ((unsigned long long)s.nnz << 32) | s.nno;
  else k.primary = (unsigned long long)__double_as_longlong(s.g2);  // g2 >= 0: order preserving
  k.index = index;
  return k;
}

constexpr int kThreads = 128;

template <int M, int K, int N>
struct MaxDim2 {
  static constexpr int d = (M > K ? (M > N ? M : N) : (K > N ? K : N));
  static constexpr int value = d * d;
};

// One candidate per thread, grid-stride over [lo,hi); per-block best to block_best[blockIdx.x].
// Dynamic shared memory: lutn doubles (sqrt table, G2 only) then the expansion scratch.
template <int M, int K, int N, int MODE, int MEASURE, int RU, bool LF, bool PACK>
__global__ void __launch_bounds__(kThreads, (PACK && M * K * N >= 84) ? (MEASURE == PLO_MEASURE_NNZ ? 4 : 3) : 0) orbit_sweep_kernel(int r, int3 den, unsigned long long seed, unsigned long long lo,
                                                                unsigned long long hi, int lutn, Key* __restrict__ block_best) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  double* lut = reinterpret_cast<double*>(dyn_smem);
  int* scr = reinterpret_cast<int*>(dyn_smem + (size_t)lutn * sizeof(double));
  __shared__ Key red[32];
  constexpr bool TAB = PACK && M == 2 && K == 2 && N == 2;
  __shared__ __align__(16) int z2tab[TAB ? kZ2Count * kZ2Stride : 4];
  if (TAB) build_zoi2_table<MODE>(z2tab);
  if (MEASURE == PLO_MEASURE_G2) {
    for (int e = threadIdx.x; e < lutn; e += kThreads) lut[e] = sqrt((double)e);
  }
  __syncthreads();
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kThreads + threadIdx.x; idx < hi; idx += stride) {
    constexpr bool SPLIT = PACK && !TAB && MEASURE == PLO_MEASURE_NNZ && RU == 0;
    Score s;
    if (SPLIT) s = score_candidate_nnz_split<M, K, N, MODE>(c_lrp, r, den, seed, idx, scr + threadIdx.x, kThreads);
    else s = score_candidate<M, K, N, MODE, MEASURE, RU, LF, PACK, TAB>(c_lrp, r, den, seed, idx, scr + threadIdx.x, kThreads, lut, lutn, z2tab);
    const Key k = make_key<MEASURE>(s, idx);
    if (k.primary < best.primary) best = k;  // indices visited in increasing order: strict '<' keeps the first
    surv_emit(k);
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// Reduce the per-block keys, re-evaluate the winner with every measure, write the result record.
template <int M, int K, int N, int MODE>
__global__ void __launch_bounds__(kThreads) orbit_final_kernel(int r, int3 den, unsigned long long seed, int nblocks, int measure,
                                                                double inv_den, const Key* __restrict__ block_best,
                                                                plo_orbit_best* __restrict__ out) {
  __shared__ int scr[MaxDim2<M, K, N>::value * kThreads];
  __shared__ Key red[32];
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (int b = threadIdx.x; b < nblocks; b += kThreads) {
    const Key k = block_best[b];
    if (key_less(k, best)) best = k;
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) {
    plo_orbit_best o;
    o.index = best.index;
    o.nnz = 0; o.nno = 0; o.score = 0.0;
    if (best.index != ~0ull) {
      const Score s = score_candidate<M, K, N, MODE, MEASURE_BOTH>(c_lrp, r, den, seed, best.index, scr, kThreads);
      o.nnz = s.nnz; o.nno = s.nno;
      o.score = (measure == PLO_MEASURE_G2) ? s.g2 * inv_den : (double)s.nnz;
    }
    *out = o;
  }
}

// Survivor compaction: every candidate whose score does not exceed a threshold is appended to a device buffer.  The survivors of a
// warp take consecutive 32-byte records (one atomicAdd per warp, two 16-byte stores per survivor): coalesced, vectorised, in no
// particular order -- the host sorts by index.  `count` keeps counting past `cap` so that the caller learns the size it needs.
struct Sink {
  uint4* rec;                 // {index lo, index hi, nnz, nno} {score bits lo, score bits hi, 0, 0}
  unsigned long long* count;
  unsigned long long cap;
  unsigned long long thr_key;  // sparsity: (nnz << 32) | nno
  double thr_score;            // growth factor
  int measure;
};
__device__ __forceinline__ void sink_emit(const Sink& sk, bool valid, unsigned long long idx, uint32_t nnz, uint32_t nno, double score) {
  // called by all 32 lanes of a warp (warp-uniform loops below)
  const bool pass = valid && (sk.measure == PLO_MEASURE_G2 ? score <= sk.thr_score : ((((unsigned long long)nnz) << 32) | nno) <= sk.thr_key);
  const unsigned mask = __ballot_sync(0xffffffffu, pass);
  if (mask == 0u) return;
  const int lane = threadIdx.x & 31;
  unsigned long long base = 0;
  if (lane == __ffs(mask) - 1) base = atomicAdd(sk.count, (unsigned long long)__popc(mask));
  base = __shfl_sync(0xffffffffu, base, __ffs(mask) - 1);
  if (pass) {
    const unsigned long long pos = base + __popc(mask & ((1u << lane) - 1u));
    if (pos < sk.cap) {
      const unsigned long long sb = (unsigned long long)__double_as_longlong(score);
      sk.rec[2 * pos] = make_uint4((unsigned)idx, (unsigned)(idx >> 32), nnz, nno);
      sk.rec[2 * pos + 1] = make_uint4((unsigned)sb, (unsigned)(sb >> 32), 0u, 0u);
    }
  }
}

// Per-candidate table and/or survivor compaction (both measures of every candidate; warp-uniform loop: whole warps step together).
template <int M, int K, int N, int MODE>
__global__ void __launch_bounds__(kThreads) orbit_table_kernel(int r, int3 den, unsigned long long seed, unsigned long long lo,
                                                                unsigned long long hi, double inv_den,
                                                                uint32_t* __restrict__ nnz, uint32_t* __restrict__ nno,
                                                                double* __restrict__ g2, Sink sink) {
  __shared__ int scr[MaxDim2<M, K, N>::value * kThreads];
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  const int lane = threadIdx.x & 31;
  for (unsigned long long wb = lo + (unsigned long long)blockIdx.x * kThreads + (threadIdx.x - lane); wb < hi; wb += stride) {
    const unsigned long long idx = wb + lane;
    const bool valid = idx < hi;
    Score s;
    s.nnz = 0; s.nno = 0; s.g2 = 0.0;
    if (valid) {
      s = score_candidate<M, K, N, MODE, MEASURE_BOTH>(c_lrp, r, den, seed, idx, scr + threadIdx.x, kThreads);
      if (nnz) nnz[idx - lo] = s.nnz;
      if (nno) nno[idx - lo] = s.nno;
      if (g2) g2[idx - lo] = s.g2 * inv_den;
    }
    if (sink.rec) sink_emit(sink, valid, idx, s.nnz, s.nno, s.g2 * inv_den);
  }
}

// Both measures of a LIST of candidates (the survivors of a sweep, sorted by index): one record of 32 bytes each, two 16-byte stores.
template <int M, int K, int N, int MODE>
__global__ void __launch_bounds__(kThreads) orbit_gather_kernel(int r, int3 den, unsigned long long seed, const unsigned long long* __restrict__ list,
                                                                 unsigned long long count, double inv_den, uint4* __restrict__ rec) {
  __shared__ int scr[MaxDim2<M, K, N>::value * kThreads];
  for (unsigned long long t = (unsigned long long)blockIdx.x * kThreads + threadIdx.x; t < count; t += (unsigned long long)gridDim.x * kThreads) {
    const unsigned long long idx = list[t];
    const Score sc = score_candidate<M, K, N, MODE, MEASURE_BOTH>(c_lrp, r, den, seed, idx, scr + threadIdx.x, kThreads);
    const unsigned long long sb = (unsigned long long)__double_as_longlong(sc.g2 * inv_den);
    rec[2 * t] = make_uint4((unsigned)idx, (unsigned)(idx >> 32), sc.nnz, sc.nno);
    rec[2 * t + 1] = make_uint4((unsigned)sb, (unsigned)(sb >> 32), 0u, 0u);
  }
}

// ---------------------------------------------------------------------------
// Orbit sweep over Z/pZ  (`orbiter -m p`: FMatrix L(BL,FF) ... src/orbiter.cpp:232-234, 419-426;
// the whole search then runs in the field, measure = sparsity, Orbiter<0>).
// L, R, P^T hold residues in [0,p), p < 2^31.  U, V, W and their inverses are small integers,
// so a transformed entry is an integer combination of residues: both stages of the product are
// accumulated exactly in 64 bits (|.| < 2^31 . 2^8 . 2^8) and reduced ONCE, by a Barrett
// reduction of (value + bias) with bias a multiple of p above 2^48.
// ---------------------------------------------------------------------------
struct ModP {
  unsigned int p;
  unsigned long long M64;   // floor((2^64-1)/p)
  unsigned long long bias;  // multiple of p, >= 2^48
};
__host__ __device__ __forceinline__ unsigned int modp_reduce(long long v, const ModP& mp) {
  const unsigned long long x = (unsigned long long)(v + (long long)mp.bias);
#ifdef __CUDA_ARCH__
  const unsigned long long q = __umul64hi(x, mp.M64);
#else
  const unsigned long long q = (unsigned long long)(((unsigned __int128)x * mp.M64) >> 64);
#endif
  unsigned long long r = x - q * mp.p;
  if (r >= mp.p) r -= mp.p;
  if (r >= mp.p) r -= mp.p;
  return (unsigned int)r;
}
template <int RA, int CA, bool TL, bool TR>
__host__ __device__ __forceinline__ void transform_row_modp(const int* __restrict__ A, const int* Lm, const int* Rm, const ModP& mp, Acc& acc) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A[e];
#pragma unroll
  for (int x = 0; x < RA; ++x) {
    long long X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      long long s = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) s += (long long)(TL ? Lm[i * RA + x] : Lm[x * RA + i]) * (long long)a[i * CA + j];
      X[j] = s;
    }
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      long long s = 0;
#pragma unroll
      for (int j = 0; j < CA; ++j) s += X[j] * (long long)(TR ? Rm[y * CA + j] : Rm[j * CA + y]);
      const unsigned int v = modp_reduce(s, mp);
      acc.nnz += (v != 0u);
      acc.nno += (v != 0u) & (v != 1u) & (v != mp.p - 1u);  // isAbsOne in the field
    }
  }
}
template <int M, int K, int N, int MODE>
__host__ __device__ __forceinline__ Score score_candidate_modp(const int* __restrict__ lrp, int r, const ModP& mp, unsigned long long seed,
                                                               unsigned long long index, volatile int* scr, int stride) {
  Digits<MODE> ds(seed, index);
  const Zoi zu = decode_zoi<M, MODE>(ds);
  const Zoi zv = decode_zoi<K, MODE>(ds);
  const Zoi zw = decode_zoi<N, MODE>(ds);
  int U[M * M], Ui[M * M], V[K * K], Vi[K * K], W[N * N], Wi[N * N];
  expand_zoi<M, false>(zu, U, scr, stride);
  expand_zoi<M, true>(zu, Ui, scr, stride);
  expand_zoi<K, false>(zv, V, scr, stride);
  expand_zoi<K, true>(zv, Vi, scr, stride);
  expand_zoi<N, false>(zw, W, scr, stride);
  expand_zoi<N, true>(zw, Wi, scr, stride);
  const int* Lc = lrp;
  const int* Rc = lrp + r * M * K;
  const int* Pc = Rc + r * K * N;
  Acc acc;
  acc.nnz = acc.nno = acc.sq = 0;
  for (int l = 0; l < r; ++l) {
    transform_row_modp<M, K, true, false>(Lc + l * M * K, Ui, V, mp, acc);   // U^-T A V
    transform_row_modp<K, N, false, false>(Rc + l * K * N, Vi, W, mp, acc);  // V^-1 B W
    transform_row_modp<M, N, false, true>(Pc + l * M * N, U, Wi, mp, acc);   // U C W^-T
  }
  Score sc;
  sc.nnz = (uint32_t)acc.nnz; sc.nno = (uint32_t)acc.nno; sc.g2 = 0.0;
  return sc;
}

template <int M, int K, int N, int MODE>
__global__ void __launch_bounds__(kThreads) orbit_modp_kernel(int r, ModP mp, unsigned long long seed, unsigned long long lo, unsigned long long hi,
                                                               Key* __restrict__ block_best, uint32_t* __restrict__ tnnz, uint32_t* __restrict__ tnno) {
  __shared__ int scr[MaxDim2<M, K, N>::value * kThreads];
  __shared__ Key red[32];
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kThreads + threadIdx.x; idx < hi; idx += stride) {
    const Score s = score_candidate_modp<M, K, N, MODE>(c_lrp, r, mp, seed, idx, scr + threadIdx.x, kThreads);
    if (tnnz) tnnz[idx - lo] = s.nnz;
    if (tnno) tnno[idx - lo] = s.nno;
    const Key k = make_key<PLO_MEASURE_NNZ>(s, idx);
    if (k.primary < best.primary) best = k;
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// ---------------------------------------------------------------------------
// Four-lane growth-factor path for small magnitudes (every transformed entry in [-127, 127]: integer-coefficient algorithms such as
// Strassen / Winograd / Laderman).  Two rows x0,x1 of the left factor travel at 16-bit spacing (pack_left) AND two Hopcroft-Musinski
// rows l,l+1 of the input at 8-bit spacing (host-packed c_lrp2), so one IMAD carries four products:
//   (l0 + 2^16 l1)(a0 + 2^8 a1) = l0a0 + 2^8 l0a1 + 2^16 l1a0 + 2^24 l1a1   ->   lanes (x0,l) (x0,l+1) (x1,l) (x1,l+1).
// v + 0x80808080 absorbs the borrows bottom-up, ^ 0x80808080 leaves four signed bytes; the squares of the two lanes that belong to
// row l (bytes 0,2) and to row l+1 (bytes 1,3) are accumulated by one dp4a each.  Same doubles, same summation order as the other
// paths: bit-identical G2.
// ---------------------------------------------------------------------------
template <int RA, int CA, bool TR>
__device__ __forceinline__ void transform_pair_packed8(const int* __restrict__ A2, const int* LmP, const int* Rm, int& sq0, int& sq1) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A2[e];
#pragma unroll
  for (int xp = 0; xp < (RA + 1) / 2; ++xp) {
    int X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      int s = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) s += LmP[xp * RA + i] * a[i * CA + j];
      X[j] = s;
    }
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      int v = 0;
#pragma unroll
      for (int j = 0; j < CA; ++j) v += X[j] * (TR ? Rm[y * CA + j] : Rm[j * CA + y]);
      const unsigned x = ((unsigned)v + 0x80808080u) ^ 0x80808080u;  // ptxas folds the bias into the first multiply-add
      sq0 = __dp4a((int)x, (int)(x & 0x00FF00FFu), sq0);
      sq1 = __dp4a((int)x, (int)(x & 0xFF00FF00u), sq1);
    }
  }
}

// The same with a triangular right factor (see "Triangular right factors"): LOWER = false for X.M (sum over i < y), true for X.M^-T
// (sum over j > y).  scr = this thread's scratch column, poff[i] = offset of X[P[i]] in it.
template <int RA, int CA, bool LOWER>
__device__ __forceinline__ void transform_pair_packed8_tri(const int* __restrict__ A2, const int* LmP, const int* tri, const int* poff, volatile int* scr,
                                                           int& sq0, int& sq1) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A2[e];
#pragma unroll
  for (int xp = 0; xp < (RA + 1) / 2; ++xp) {
    int X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      int acc = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) acc += LmP[xp * RA + i] * a[i * CA + j];
      scr[j * kThreads] = acc;
    }
#pragma unroll
    for (int i = 0; i < CA; ++i) X[i] = scr[poff[i]];
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      int v = X[y];
      if (!LOWER) {
#pragma unroll
        for (int i = 0; i < y; ++i) v += X[i] * tri[tri_index<CA>(i, y)];
      } else {
#pragma unroll
        for (int j = y + 1; j < CA; ++j) v += X[j] * tri[tri_index<CA>(y, j)];
      }
      const unsigned x = ((unsigned)v + 0x80808080u) ^ 0x80808080u;
      sq0 = __dp4a((int)x, (int)(x & 0x00FF00FFu), sq0);
      sq1 = __dp4a((int)x, (int)(x & 0xFF00FF00u), sq1);
    }
  }
}

// 3x3 zoi matrices: 6.6.8.27 = 7776 per factor -- too many for shared memory, but one table per plan in global memory (1.5 MB,
// L2-resident) still replaces decode + expansion + inverse + packing (~450 instructions per candidate) by 15 128-bit loads.
// Entry = 12 chunks of 16 bytes: M (9 ints, 3 chunks) | M^-1 (3) | pack_left<T>(M^-1) (6 ints, 2) | pack_left(M) (2) | pack_left(M^-1) (2).
constexpr int kZ3Count = 7776, kZ3Chunks = 12;
template <int MODE>
__global__ void __launch_bounds__(kThreads) zoi3_table_kernel(int4* __restrict__ tab) {
  __shared__ int scr0[9 * kThreads];
  const int e = blockIdx.x * kThreads + threadIdx.x;
  if (e >= kZ3Count) return;
  volatile int* scr = scr0 + threadIdx.x;
  RawDigits<MODE> ds((uint32_t)e, (uint32_t)kZ3Count);
  const Zoi z = decode_zoi<3, MODE, RawDigits<MODE>>(ds);
  int Mx[9], Mi[9], pit[6], pm[6], pi[6];
  expand_zoi<3, false>(z, Mx, scr, kThreads);
  expand_zoi<3, true>(z, Mi, scr, kThreads);
  pack_left<3, true>(Mi, pit);
  pack_left<3, false>(Mx, pm);
  pack_left<3, false>(Mi, pi);
  int4* t = tab + (size_t)e * kZ3Chunks;
  t[0] = make_int4(Mx[0], Mx[1], Mx[2], Mx[3]); t[1] = make_int4(Mx[4], Mx[5], Mx[6], Mx[7]); t[2] = make_int4(Mx[8], 0, 0, 0);
  t[3] = make_int4(Mi[0], Mi[1], Mi[2], Mi[3]); t[4] = make_int4(Mi[4], Mi[5], Mi[6], Mi[7]); t[5] = make_int4(Mi[8], 0, 0, 0);
  t[6] = make_int4(pit[0], pit[1], pit[2], pit[3]); t[7] = make_int4(pit[4], pit[5], 0, 0);
  t[8] = make_int4(pm[0], pm[1], pm[2], pm[3]); t[9] = make_int4(pm[4], pm[5], 0, 0);
  t[10] = make_int4(pi[0], pi[1], pi[2], pi[3]); t[11] = make_int4(pi[4], pi[5], 0, 0);
}
__device__ __forceinline__ void z3_load9(const int4* t, int* out) {
  const int4 a = __ldg(t), b = __ldg(t + 1), c = __ldg(t + 2);
  out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w; out[8] = c.x;
}
__device__ __forceinline__ void z3_load6(const int4* t, int* out) {
  const int4 a = __ldg(t), b = __ldg(t + 1);
  out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y;
}
// all a candidate of a 3x3x3 sweep needs from the table: pack(U^-T), pack(U), V, pack(V^-1), W, W^-1
template <int MODE>
__device__ __forceinline__ void z3_candidate(const int4* __restrict__ z3tab, Digits<MODE>& ds, int* UiTP, int* UP, int* V, int* ViP, int* W, int* Wi) {
  const int4* tu = z3tab + (size_t)ds.matrix_index(kZ3Count) * kZ3Chunks;
  const int4* tv = z3tab + (size_t)ds.matrix_index(kZ3Count) * kZ3Chunks;
  const int4* tw = z3tab + (size_t)ds.matrix_index(kZ3Count) * kZ3Chunks;
  z3_load6(tu + 6, UiTP);
  z3_load6(tu + 8, UP);
  z3_load9(tv, V);
  z3_load6(tv + 10, ViP);
  z3_load9(tw, W);
  z3_load9(tw + 3, Wi);
}

template <int M, int K, int N, int MODE, int RU, bool LF, bool TAB>
__device__ __forceinline__ Key sweep8_loop(int r, unsigned long long seed, unsigned long long lo, unsigned long long hi, int lutn, const double* lut,
                                           volatile int* scr, const int* z2tab, int npair, const int* L2, const int* R2, const int* P2,
                                           const int4* __restrict__ z3tab) {
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kThreads + threadIdx.x; idx < hi; idx += stride) {
    Digits<MODE> ds(seed, idx);
    constexpr bool TRIW = N >= 5 && !TAB;  // large right factor: triangular form (only S(S-1)/2 of the N*N slots below are used then)
    int V[K * K], W[TRIW ? N * (N - 1) / 2 : N * N], Wi[TRIW ? N * (N - 1) / 2 : N * N], wpoff[TRIW ? N : 1];
    int UiTP[((M + 1) / 2) * M], ViP[((K + 1) / 2) * K], UP[((M + 1) / 2) * M];
    if (TAB) {
      const int* tu = z2tab + ds.matrix_index(kZ2Count) * kZ2Stride;
      const int* tv = z2tab + ds.matrix_index(kZ2Count) * kZ2Stride;
      const int* tw = z2tab + ds.matrix_index(kZ2Count) * kZ2Stride;
      int both[4];
      z2_load4(tu + 8, both);
      UiTP[0] = both[0]; UiTP[1] = both[1]; UP[0] = both[2]; UP[1] = both[3];
      z2_load4(tv, V);
      z2_load2(tv + 12, ViP);
      z2_load4(tw, W);
      z2_load4(tw + 4, Wi);
    } else if (M == 3 && K == 3 && N == 3 && z3tab != nullptr) {
      z3_candidate<MODE>(z3tab, ds, UiTP, UP, V, ViP, W, Wi);
    } else {
      const Zoi zu = decode_zoi<M, MODE>(ds);
      const Zoi zv = decode_zoi<K, MODE>(ds);
      const Zoi zw = decode_zoi<N, MODE>(ds);
      int U[M * M], Ui[M * M], Vi[K * K];
      expand_zoi<M, false>(zu, U, scr, kThreads);
      expand_zoi<M, true>(zu, Ui, scr, kThreads);
      expand_zoi<K, false>(zv, V, scr, kThreads);
      expand_zoi<K, true>(zv, Vi, scr, kThreads);
      if (TRIW) {  // W and W^-T as triangular right factors: 2 x 21 registers instead of 2 x 49 for a 7x7 factor
        zoi_tri<N, false>(zw, W);
        zoi_tri<N, true>(zw, Wi);
        zoi_perm_offsets<N>(zw, kThreads, wpoff);
      } else {
        expand_zoi<N, false>(zw, W, scr, kThreads);
        expand_zoi<N, true>(zw, Wi, scr, kThreads);
      }
      pack_left<M, true>(Ui, UiTP);
      pack_left<K, false>(Vi, ViP);
      pack_left<M, false>(U, UP);
    }
    double g2 = 0.0;
#pragma unroll(RU > 0 ? (RU + 1) / 2 : 1)
    for (int q = 0; q < npair; ++q) {
      int sL0 = 0, sL1 = 0, sR0 = 0, sR1 = 0, sP0 = 0, sP1 = 0;
      transform_pair_packed8<M, K, false>(L2 + q * M * K, UiTP, V, sL0, sL1);   // U^-T A V
      if (TRIW) {
        transform_pair_packed8_tri<K, N, false>(R2 + q * K * N, ViP, W, wpoff, scr, sR0, sR1);    // V^-1 B W
        transform_pair_packed8_tri<M, N, true>(P2 + q * M * N, UP, Wi, wpoff, scr, sP0, sP1);     // U C W^-T
      } else {
      transform_pair_packed8<K, N, false>(R2 + q * K * N, ViP, W, sR0, sR1);    // V^-1 B W
      transform_pair_packed8<M, N, true>(P2 + q * M * N, UP, Wi, sP0, sP1);     // U C W^-T
      }
      // growthfactor.cpp:117-125, rows in order, no FMA contraction
      // table lookup; a row norm^2 beyond the table (worst-case bound larger than the 4096 entries kept) takes the out-of-line sqrt
      auto root = [&](int sq) { return (LF || sq < lutn) ? lut[sq] : slow_isqrt(sq); };
      g2 = __dadd_rn(g2, __dmul_rn(__dmul_rn(root(sL0), root(sR0)), root(sP0)));
      if (2 * q + 1 < (RU > 0 ? RU : r)) g2 = __dadd_rn(g2, __dmul_rn(__dmul_rn(root(sL1), root(sR1)), root(sP1)));
    }
    Key k;
    k.primary = (unsigned long long)__double_as_longlong(g2);
    k.index = idx;
    if (k.primary < best.primary) best = k;
    surv_emit(k);
  }
  return best;
}

template <int M, int K, int N, int MODE, int RU>
__global__ void __launch_bounds__(kThreads, (M * K * N >= 84) ? PLO_SWEEP8_MINB : 1) orbit_sweep8_kernel(int r, unsigned long long seed, unsigned long long lo, unsigned long long hi, int lutn, int lutfull,
                                                                 Key* __restrict__ block_best, const int4* __restrict__ z3tab) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  double* lut = reinterpret_cast<double*>(dyn_smem);
  int* scr0 = reinterpret_cast<int*>(dyn_smem + (size_t)lutn * sizeof(double));
  __shared__ Key red[32];
  constexpr bool TAB = M == 2 && K == 2 && N == 2;
  __shared__ __align__(16) int z2tab[TAB ? kZ2Count * kZ2Stride : 4];
  if (TAB) build_zoi2_table<MODE>(z2tab);
  for (int e = threadIdx.x; e < lutn; e += kThreads) lut[e] = sqrt((double)e);
  __syncthreads();
  volatile int* scr = scr0 + threadIdx.x;
  const int npair = RU > 0 ? (RU + 1) / 2 : (r + 1) / 2;
  const int* L2 = c_lrp2;
  const int* R2 = L2 + npair * M * K;
  const int* P2 = R2 + npair * K * N;
  Key best;
  if (lutfull) best = sweep8_loop<M, K, N, MODE, RU, true, TAB>(r, seed, lo, hi, lutn, lut, scr, z2tab, npair, L2, R2, P2, z3tab);
  else best = sweep8_loop<M, K, N, MODE, RU, false, TAB>(r, seed, lo, hi, lutn, lut, scr, z2tab, npair, L2, R2, P2, z3tab);
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// ---------------------------------------------------------------------------
// Four-lane SPARSITY kernel (same packing as orbit_sweep8_kernel: every transformed entry in [-127, 127], denominators < 128).
// A word w = v + 0x80808080 holds four biased lanes; VABSDIFF4.U8(w, 0x80808080) is |lane| per byte (<= 127), and for a word a of
// bytes <= 127 the bytes that differ from a constant c are the bit-7 positions of ((a ^ c) + 0x7f7f7f7f): non-zero lanes with c = 0,
// lanes with |y| != den with c = den.  The marks are summed as byte counters (LEA.HI: acc + (mask >> 7)), flushed into 32-bit
// totals by one dp4a per pair of rows (at most 3.ceil(RA/2).CA <= 63 marks per byte between flushes).  Phantom lanes (odd RA, odd r) are
// zero: they add nothing to nnz and count as "!= den".   nno = nnz - #(|y| == den) = nnz - (lanes - #(|y| != den)).
// Half the IMADs of the two-lane kernels at the same number of classification instructions per lane.
// ---------------------------------------------------------------------------
template <int RA, int CA, bool TR>
__device__ __forceinline__ void transform_pair_count8(const int* __restrict__ A2, const int* LmP, const int* Rm, unsigned dd, unsigned& cz, unsigned& cd) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A2[e];
#pragma unroll
  for (int xp = 0; xp < (RA + 1) / 2; ++xp) {
    int X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      int s = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) s += LmP[xp * RA + i] * a[i * CA + j];
      X[j] = s;
    }
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      int v = 0;
#pragma unroll
      for (int j = 0; j < CA; ++j) v += X[j] * (TR ? Rm[y * CA + j] : Rm[j * CA + y]);
      const unsigned ab = __vabsdiffu4((unsigned)v + 0x80808080u, 0x80808080u);
      // acc + (mask >> 7) as ONE multiply-high-add (mask . 2^25 >> 32): the fma-heavy pipe has room here, the alu pipe does not
      asm("mad.hi.u32 %0, %1, 0x02000000, %0;" : "+r"(cz) : "r"((ab + 0x7F7F7F7Fu) & 0x80808080u));
      asm("mad.hi.u32 %0, %1, 0x02000000, %0;" : "+r"(cd) : "r"(((ab ^ dd) + 0x7F7F7F7Fu) & 0x80808080u));
    }
  }
}

template <int RA, int CA, bool LOWER>
__device__ __forceinline__ void transform_pair_count8_tri(const int* __restrict__ A2, const int* LmP, const int* tri, const int* poff, volatile int* scr,
                                                          unsigned dd, unsigned& cz, unsigned& cd) {
  int a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A2[e];
#pragma unroll
  for (int xp = 0; xp < (RA + 1) / 2; ++xp) {
    int X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      int acc = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) acc += LmP[xp * RA + i] * a[i * CA + j];
      scr[j * kThreads] = acc;
    }
#pragma unroll
    for (int i = 0; i < CA; ++i) X[i] = scr[poff[i]];
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      int v = X[y];
      if (!LOWER) {
#pragma unroll
        for (int i = 0; i < y; ++i) v += X[i] * tri[tri_index<CA>(i, y)];
      } else {
#pragma unroll
        for (int j = y + 1; j < CA; ++j) v += X[j] * tri[tri_index<CA>(y, j)];
      }
      const unsigned ab = __vabsdiffu4((unsigned)v + 0x80808080u, 0x80808080u);
      asm("mad.hi.u32 %0, %1, 0x02000000, %0;" : "+r"(cz) : "r"((ab + 0x7F7F7F7Fu) & 0x80808080u));
      asm("mad.hi.u32 %0, %1, 0x02000000, %0;" : "+r"(cd) : "r"(((ab ^ dd) + 0x7F7F7F7Fu) & 0x80808080u));
    }
  }
}

template <int M, int K, int N, int MODE>
__global__ void __launch_bounds__(kThreads, (M * K * N >= 84) ? PLO_SWEEPN8_MINB : 1) orbit_sweepn8_kernel(int r, int3 den, unsigned long long seed, unsigned long long lo, unsigned long long hi,
                                                                  Key* __restrict__ block_best, const int4* __restrict__ z3tab) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  int* scr0 = reinterpret_cast<int*>(dyn_smem);
  __shared__ Key red[32];
  volatile int* scr = scr0 + threadIdx.x;
  const int npair = (r + 1) / 2;
  const int* L2 = c_lrp2;
  const int* R2 = L2 + npair * M * K;
  const int* P2 = R2 + npair * K * N;
  const unsigned dL = (unsigned)den.x * 0x01010101u, dR = (unsigned)den.y * 0x01010101u, dP = (unsigned)den.z * 0x01010101u;
  constexpr int lanes = 4 * (((M + 1) / 2) * K + ((K + 1) / 2) * N + ((M + 1) / 2) * N);  // per pair of rows, phantom lanes included
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kThreads + threadIdx.x; idx < hi; idx += stride) {
    Digits<MODE> ds(seed, idx);
    if (M * K * N >= 84) {
      // Large shapes (3x4x7: W and W^-T alone are 98 registers): the counts are sums over the three products, so the rows of L, then
      // of R, then of P are swept with only the two matrices of that product live -- 222 -> 128 registers, 2 -> 4 blocks per SM.
      // The byte counters are flushed per pair of rows and phase (at most ceil(RA/2).CA <= 14 marks per byte in between).
      const Zoi zu = decode_zoi<M, MODE>(ds);
      const Zoi zv = decode_zoi<K, MODE>(ds);
      const Zoi zw = decode_zoi<N, MODE>(ds);
      unsigned z = 0, d = 0;
      {
        int Ui[M * M], V[K * K], UiTP[((M + 1) / 2) * M];
        expand_zoi<M, true>(zu, Ui, scr, kThreads);
        pack_left<M, true>(Ui, UiTP);
        expand_zoi<K, false>(zv, V, scr, kThreads);
#pragma unroll 1
        for (int q = 0; q < npair; ++q) {
          unsigned cz = 0, cd = 0;
          transform_pair_count8<M, K, false>(L2 + q * M * K, UiTP, V, dL, cz, cd);   // U^-T A V
          z = __dp4a(cz, 0x01010101u, z);
          d = __dp4a(cd, 0x01010101u, d);
        }
      }
      int wpoff[N];
      zoi_perm_offsets<N>(zw, kThreads, wpoff);
      {
        int Vi[K * K], Wt[N * (N - 1) / 2], ViP[((K + 1) / 2) * K];
        expand_zoi<K, true>(zv, Vi, scr, kThreads);
        pack_left<K, false>(Vi, ViP);
        zoi_tri<N, false>(zw, Wt);
#pragma unroll 1
        for (int q = 0; q < npair; ++q) {
          unsigned cz = 0, cd = 0;
          transform_pair_count8_tri<K, N, false>(R2 + q * K * N, ViP, Wt, wpoff, scr, dR, cz, cd);    // V^-1 B W, W as a triangular factor
          z = __dp4a(cz, 0x01010101u, z);
          d = __dp4a(cd, 0x01010101u, d);
        }
      }
      {
        int U[M * M], Wit[N * (N - 1) / 2], UP[((M + 1) / 2) * M];
        expand_zoi<M, false>(zu, U, scr, kThreads);
        pack_left<M, false>(U, UP);
        zoi_tri<N, true>(zw, Wit);
#pragma unroll 1
        for (int q = 0; q < npair; ++q) {
          unsigned cz = 0, cd = 0;
          transform_pair_count8_tri<M, N, true>(P2 + q * M * N, UP, Wit, wpoff, scr, dP, cz, cd);     // U C W^-T, W^-T as a triangular factor
          z = __dp4a(cz, 0x01010101u, z);
          d = __dp4a(cd, 0x01010101u, d);
        }
      }
      Key k;
      k.primary = ((unsigned long long)z << 32) | (unsigned long long)(z - ((unsigned)(npair * lanes) - d));
      k.index = idx;
      if (k.primary < best.primary) best = k;
      surv_emit(k);
      continue;
    }
    int V[K * K], W[N * N], Wi[N * N];
    int UiTP[((M + 1) / 2) * M], ViP[((K + 1) / 2) * K], UP[((M + 1) / 2) * M];
    if (M == 3 && K == 3 && N == 3 && z3tab != nullptr) {
      z3_candidate<MODE>(z3tab, ds, UiTP, UP, V, ViP, W, Wi);
    } else {
      const Zoi zu = decode_zoi<M, MODE>(ds);
      const Zoi zv = decode_zoi<K, MODE>(ds);
      const Zoi zw = decode_zoi<N, MODE>(ds);
      int U[M * M], Ui[M * M], Vi[K * K];
      expand_zoi<M, false>(zu, U, scr, kThreads);
      expand_zoi<M, true>(zu, Ui, scr, kThreads);
      expand_zoi<K, false>(zv, V, scr, kThreads);
      expand_zoi<K, true>(zv, Vi, scr, kThreads);
      expand_zoi<N, false>(zw, W, scr, kThreads);
      expand_zoi<N, true>(zw, Wi, scr, kThreads);
      pack_left<M, true>(Ui, UiTP);
      pack_left<K, false>(Vi, ViP);
      pack_left<M, false>(U, UP);
    }
    unsigned z = 0, d = 0;
#pragma unroll 1
    for (int q = 0; q < npair; ++q) {
      unsigned cz = 0, cd = 0;  // byte counters of this pair of rows
      transform_pair_count8<M, K, false>(L2 + q * M * K, UiTP, V, dL, cz, cd);   // U^-T A V
      transform_pair_count8<K, N, false>(R2 + q * K * N, ViP, W, dR, cz, cd);    // V^-1 B W
      transform_pair_count8<M, N, true>(P2 + q * M * N, UP, Wi, dP, cz, cd);     // U C W^-T
      z = __dp4a(cz, 0x01010101u, z);
      d = __dp4a(cd, 0x01010101u, d);
    }
    Key k;
    k.primary = ((unsigned long long)z << 32) | (unsigned long long)(z - ((unsigned)(npair * lanes) - d));
    k.index = idx;
    if (k.primary < best.primary) best = k;
    surv_emit(k);
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// ---------------------------------------------------------------------------
// 2x2x2, r = 7: every factor pair scored by its classes.  Each row measure of each product depends on the two factors of that
// product through their classes only (see zoi2_cl / zoi2_cr):
//   L rows (U^-T A_l V) on (cl(U), cr(V)),   R rows (V^-1 B_l W) on (cr(V), cr(W)),   P rows (U C_l W^-T) on (cl(U), cr(W)),
// 36 pairs per product.  Each block scores the 3 x 36 pairs once, exactly in int32 from c_lrp on the lowest-numbered matrix of each
// class, and a candidate then reads three records.  Class words: one 16-bit word per matrix number, 6.cl | cr << 8 (96 bytes in
// 24 banks: conflict-free).  Records are kept in R replicas, replica c at byte c . 128 / R of a 128-byte slot, and lane t reads
// replica t mod R: the lanes of a wavefront never collide, whatever their class pairs.
// ---------------------------------------------------------------------------
constexpr int kXThreads = 512, kXRows = 7, kZ2Pairs = kZ2Classes * kZ2Classes;

// The class word of every matrix number.
template <int MODE>
__device__ __forceinline__ void build_zoi2_classes(unsigned short* cls) {
  for (int e = threadIdx.x; e < kZ2Count; e += blockDim.x) {
    RawDigits<MODE> ds((uint32_t)e, (uint32_t)kZ2Count);
    const Zoi z = decode_zoi<2, MODE, RawDigits<MODE>>(ds);
    cls[e] = (unsigned short)(kZ2Classes * zoi2_cl(z) | zoi2_cr(z) << 8);
  }
}

// The kXRows row measures of class pair `item` in [0, 3 . 36): product item / 36 (0 = L, 1 = R, 2 = P), left class (item % 36) / 6,
// right class (item % 36) % 6.  `cls` = build_zoi2_classes, complete.
template <int MODE, int MEASURE>
__device__ __forceinline__ void zoi2_pair_rows(int item, const unsigned short* cls, int3 den, Acc* acc) {
  const int prod = item / kZ2Pairs, c1 = item % kZ2Pairs / kZ2Classes, c2 = item % kZ2Classes;
  // the lowest-numbered matrix of a class: first factor of the product by cl (L, P) or cr (R), second factor by cr
  int e1 = 0, e2 = 0;
  while (prod == 1 ? cls[e1] >> 8 != c1 : (cls[e1] & 255) != kZ2Classes * c1) ++e1;
  while (cls[e2] >> 8 != c2) ++e2;
  RawDigits<MODE> d1((uint32_t)e1, (uint32_t)kZ2Count), d2((uint32_t)e2, (uint32_t)kZ2Count);
  const Zoi z1 = decode_zoi<2, MODE, RawDigits<MODE>>(d1), z2 = decode_zoi<2, MODE, RawDigits<MODE>>(d2);
  int A[4], Ai[4], B[4], Bi[4];
  expand_zoi<2, false>(z1, A, nullptr, 0);
  expand_zoi<2, true>(z1, Ai, nullptr, 0);
  expand_zoi<2, false>(z2, B, nullptr, 0);
  expand_zoi<2, true>(z2, Bi, nullptr, 0);
  const int* Lc = c_lrp;
  const int* Rc = Lc + kXRows * 4;
  const int* Pc = Rc + kXRows * 4;
#pragma unroll
  for (int l = 0; l < kXRows; ++l) {
    acc[l].nnz = acc[l].nno = acc[l].sq = 0;
    if (prod == 0) transform_row<2, 2, true, false, MEASURE>(Lc + l * 4, Ai, B, den.x, acc[l]);        // U^-T A V
    else if (prod == 1) transform_row<2, 2, false, false, MEASURE>(Rc + l * 4, Ai, B, den.y, acc[l]);  // V^-1 B W
    else transform_row<2, 2, false, true, MEASURE>(Pc + l * 4, A, Bi, den.z, acc[l]);                   // U C W^-T
  }
}

// Shared-memory loads from a 32-bit shared-window address kept in a register: one address instruction per lookup (nvcc otherwise
// re-adds the window base of the dynamic array to every data-dependent offset).
__device__ __forceinline__ double2 lds_d2(uint32_t addr) {
  double2 v;
  asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ unsigned long long lds_u64(uint32_t addr) {
  unsigned long long v;
  asm("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ int lds_u16(uint32_t addr) {
  unsigned short v;
  asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
  return v;
}

// Growth factor.  Record = sqrt((double) row norm^2) of the 7 rows + one pad: 4 chunks of 16 bytes, each in 8 replicas
// (LDS.128 = 4 wavefronts, always).  A candidate costs 3 class words and 12 LDS.128; G2 = sum over the rows, in order, of
// (sL . sR) . sP without FMA contraction (growthfactor.cpp:117-125), the same doubles as every other G2 path.
constexpr int kXRep = 8, kXRecChunks = 4;
constexpr uint32_t kXChunk = kXRep * 16, kXRec = kXRecChunks * kXChunk, kXTab = kZ2Pairs * kXRec;  // bytes
constexpr size_t kXTabBytes = 3 * (size_t)kXTab;

template <int MODE>
__global__ void __launch_bounds__(kXThreads, 2) orbit_sweep8x_kernel(unsigned long long seed, unsigned long long lo, unsigned long long hi,
                                                                      Key* __restrict__ block_best) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ Key red[32];
  __shared__ unsigned short cls[kZ2Count];
  build_zoi2_classes<MODE>(cls);
  __syncthreads();
  for (int item = threadIdx.x; item < 3 * kZ2Pairs; item += kXThreads) {
    Acc acc[kXRows];
    zoi2_pair_rows<MODE, PLO_MEASURE_G2>(item, cls, make_int3(1, 1, 1), acc);
    double s[2 * kXRecChunks];
#pragma unroll
    for (int l = 0; l < 2 * kXRecChunks; ++l) s[l] = l < kXRows ? sqrt((double)acc[l].sq) : 0.0;
    double2* rec = reinterpret_cast<double2*>(dyn_smem + (size_t)item * kXRec);
    for (int q = 0; q < kXRecChunks; ++q)
      for (int c = 0; c < kXRep; ++c) rec[q * kXRep + c] = make_double2(s[2 * q], s[2 * q + 1]);
  }
  __syncthreads();
  const uint32_t mytab = (uint32_t)__cvta_generic_to_shared(dyn_smem) + (threadIdx.x % kXRep) * 16;
  const uint32_t mycls = (uint32_t)__cvta_generic_to_shared(cls);
  const unsigned long long stride = (unsigned long long)gridDim.x * kXThreads;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kXThreads + threadIdx.x; idx < hi; idx += stride) {
    Digits<MODE, true> ds(seed, idx);
    const uint32_t eu = ds.matrix_index(kZ2Count), ev = ds.matrix_index(kZ2Count), ew = ds.matrix_index(kZ2Count);
    const uint32_t wu = lds_u16(mycls + 2 * eu), wv = lds_u16(mycls + 2 * ev), ww = lds_u16(mycls + 2 * ew);
    const uint32_t cu6 = wu & 255u, cv = wv >> 8, cw = ww >> 8;
    const uint32_t tl = mytab + (cu6 + cv) * kXRec, tr = mytab + kXTab + (kZ2Classes * cv + cw) * kXRec, tp = mytab + 2 * kXTab + (cu6 + cw) * kXRec;
    double g2 = 0.0;
#pragma unroll
    for (int q = 0; q < kXRecChunks; ++q) {
      const double2 sL = lds_d2(tl + q * kXChunk), sR = lds_d2(tr + q * kXChunk), sP = lds_d2(tp + q * kXChunk);
      g2 = __dadd_rn(g2, __dmul_rn(__dmul_rn(sL.x, sR.x), sP.x));
      if (2 * q + 1 < kXRows) g2 = __dadd_rn(g2, __dmul_rn(__dmul_rn(sL.y, sR.y), sP.y));
    }
    Key k;
    k.primary = (unsigned long long)__double_as_longlong(g2);
    k.index = idx;
    if (k.primary < best.primary) best = k;
    surv_emit(k);
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// Sparsity twin.  Record = (nnz << 32) | nno of the 7 rows of the product (nno: |y| != den among the non-zeros, den of that
// product), so the candidate's key is the sum of its three records.  8 bytes in 16 replicas (LDS.64 = 2 wavefronts, always).
constexpr int kX2Rep = 16;
constexpr uint32_t kX2Rec = kX2Rep * 8, kX2Tab = kZ2Pairs * kX2Rec;  // bytes
constexpr size_t kX2TabBytes = 3 * (size_t)kX2Tab;

template <int MODE>
__global__ void __launch_bounds__(kXThreads, 2) orbit_sweep2x_kernel(int3 den, unsigned long long seed, unsigned long long lo, unsigned long long hi,
                                                                      Key* __restrict__ block_best) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ Key red[32];
  __shared__ unsigned short cls[kZ2Count];
  build_zoi2_classes<MODE>(cls);
  __syncthreads();
  for (int item = threadIdx.x; item < 3 * kZ2Pairs; item += kXThreads) {
    Acc acc[kXRows];
    zoi2_pair_rows<MODE, PLO_MEASURE_NNZ>(item, cls, den, acc);
    unsigned nnz = 0, nno = 0;
#pragma unroll
    for (int l = 0; l < kXRows; ++l) { nnz += (unsigned)acc[l].nnz; nno += (unsigned)acc[l].nno; }
    unsigned long long* rec = reinterpret_cast<unsigned long long*>(dyn_smem + (size_t)item * kX2Rec);
    for (int c = 0; c < kX2Rep; ++c) rec[c] = ((unsigned long long)nnz << 32) | nno;
  }
  __syncthreads();
  const uint32_t mytab = (uint32_t)__cvta_generic_to_shared(dyn_smem) + (threadIdx.x % kX2Rep) * 8;
  const uint32_t mycls = (uint32_t)__cvta_generic_to_shared(cls);
  const unsigned long long stride = (unsigned long long)gridDim.x * kXThreads;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kXThreads + threadIdx.x; idx < hi; idx += stride) {
    Digits<MODE, true> ds(seed, idx);
    const uint32_t eu = ds.matrix_index(kZ2Count), ev = ds.matrix_index(kZ2Count), ew = ds.matrix_index(kZ2Count);
    const uint32_t wu = lds_u16(mycls + 2 * eu), wv = lds_u16(mycls + 2 * ev), ww = lds_u16(mycls + 2 * ew);
    const uint32_t cu6 = wu & 255u, cv = wv >> 8, cw = ww >> 8;
    Key k;
    k.primary = lds_u64(mytab + (cu6 + cv) * kX2Rec) + lds_u64(mytab + kX2Tab + (kZ2Classes * cv + cw) * kX2Rec) +
                lds_u64(mytab + 2 * kX2Tab + (cu6 + cw) * kX2Rec);
    k.index = idx;
    if (k.primary < best.primary) best = k;
    surv_emit(k);
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// ---------------------------------------------------------------------------
// Wide exact path: int32 inputs whose transforms (or squares) would leave 32 bits -- e.g. 2x2x2_7_DPS-integral-12.0662, common
// denominators ~10^9.  Both stages of the product are accumulated exactly in 64 bits (|.| < 2^31 . 2^8 . 2^8, as in the modular
// path); sparsity is classified on the exact integers; for the growth factor every entry becomes a double first
// (value / denominator, growthfactor.cpp:25-28), then square / sum / sqrt per row (:41-44, 117-125): within 1e-12 relative of the
// reference formula, not bit-identical (the reference truncates the rational -> double conversion).
// ---------------------------------------------------------------------------
struct AccW {
  int nnz, nno;
  double sq;
};
template <typename TA, int RA, int CA, bool TL, bool TR>
__host__ __device__ __forceinline__ void transform_row_wide(const TA* __restrict__ A, const int* Lm, const int* Rm, long long den, double inv_den, AccW& acc) {
  TA a[RA * CA];
#pragma unroll
  for (int e = 0; e < RA * CA; ++e) a[e] = A[e];
#pragma unroll
  for (int x = 0; x < RA; ++x) {
    long long X[CA];
#pragma unroll
    for (int j = 0; j < CA; ++j) {
      long long s = 0;
#pragma unroll
      for (int i = 0; i < RA; ++i) s += (long long)(TL ? Lm[i * RA + x] : Lm[x * RA + i]) * (long long)a[i * CA + j];
      X[j] = s;
    }
#pragma unroll
    for (int y = 0; y < CA; ++y) {
      long long s = 0;
#pragma unroll
      for (int j = 0; j < CA; ++j) s += X[j] * (long long)(TR ? Rm[y * CA + j] : Rm[j * CA + y]);
      acc.nnz += (s != 0);
      acc.nno += (s != 0) & (s != den) & (s != -den);
      const double v = (double)s * inv_den;
      acc.sq += v * v;
    }
  }
}
struct Den3 {
  long long x, y, z;
};
template <typename TA, int M, int K, int N, int MODE>
__host__ __device__ __forceinline__ Score score_candidate_wide(const TA* __restrict__ lrp, int r, Den3 den, double3 inv_den, unsigned long long seed,
                                                               unsigned long long index, volatile int* scr, int stride) {
  Digits<MODE> ds(seed, index);
  const Zoi zu = decode_zoi<M, MODE>(ds);
  const Zoi zv = decode_zoi<K, MODE>(ds);
  const Zoi zw = decode_zoi<N, MODE>(ds);
  int U[M * M], Ui[M * M], V[K * K], Vi[K * K], W[N * N], Wi[N * N];
  expand_zoi<M, false>(zu, U, scr, stride);
  expand_zoi<M, true>(zu, Ui, scr, stride);
  expand_zoi<K, false>(zv, V, scr, stride);
  expand_zoi<K, true>(zv, Vi, scr, stride);
  expand_zoi<N, false>(zw, W, scr, stride);
  expand_zoi<N, true>(zw, Wi, scr, stride);
  const TA* Lc = lrp;
  const TA* Rc = lrp + r * M * K;
  const TA* Pc = Rc + r * K * N;
  Score sc;
  sc.nnz = 0; sc.nno = 0; sc.g2 = 0.0;
  for (int l = 0; l < r; ++l) {
    AccW aL, aR, aP;
    aL.nnz = aL.nno = 0; aL.sq = 0.0;
    aR = aL; aP = aL;
    transform_row_wide<TA, M, K, true, false>(Lc + l * M * K, Ui, V, den.x, inv_den.x, aL);
    transform_row_wide<TA, K, N, false, false>(Rc + l * K * N, Vi, W, den.y, inv_den.y, aR);
    transform_row_wide<TA, M, N, false, true>(Pc + l * M * N, U, Wi, den.z, inv_den.z, aP);
    sc.nnz += (uint32_t)(aL.nnz + aR.nnz + aP.nnz);
    sc.nno += (uint32_t)(aL.nno + aR.nno + aP.nno);
    sc.g2 += (sqrt(aL.sq) * sqrt(aR.sq)) * sqrt(aP.sq);
  }
  return sc;
}
template <typename TA, int M, int K, int N, int MODE>
__global__ void __launch_bounds__(kThreads) orbit_wide_kernel(int r, Den3 den, double3 inv_den, int measure, unsigned long long seed, unsigned long long lo,
                                                               unsigned long long hi, Key* __restrict__ block_best, uint32_t* __restrict__ tnnz,
                                                               uint32_t* __restrict__ tnno, double* __restrict__ tg2, Sink sink) {
  __shared__ int scr[MaxDim2<M, K, N>::value * kThreads];
  __shared__ Key red[32];
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  const int lane = threadIdx.x & 31;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long wb = lo + (unsigned long long)blockIdx.x * kThreads + (threadIdx.x - lane); wb < hi; wb += stride) {
    const unsigned long long idx = wb + lane;
    const bool valid = idx < hi;
    Score s;
    s.nnz = 0; s.nno = 0; s.g2 = 0.0;
    if (valid) {
      s = score_candidate_wide<TA, M, K, N, MODE>(reinterpret_cast<const TA*>(c_lrp), r, den, inv_den, seed, idx, scr + threadIdx.x, kThreads);
      if (tnnz) tnnz[idx - lo] = s.nnz;
      if (tnno) tnno[idx - lo] = s.nno;
      if (tg2) tg2[idx - lo] = s.g2;
      Key k;
      k.primary = measure == PLO_MEASURE_G2 ? (unsigned long long)__double_as_longlong(s.g2) : (((unsigned long long)s.nnz << 32) | s.nno);
      k.index = idx;
      if (k.primary < best.primary) best = k;
    }
    if (sink.rec) sink_emit(sink, valid, idx, s.nnz, s.nno, s.g2);
  }
  best = block_min(best, red);
  if (threadIdx.x == 0 && block_best) block_best[blockIdx.x] = best;
}
static Sink no_sink() {
  Sink sk;
  sk.rec = nullptr; sk.count = nullptr; sk.cap = 0; sk.thr_key = 0; sk.thr_score = 0.0; sk.measure = PLO_MEASURE_NNZ;
  return sk;
}

// f(std::integral_constant<int, MODE>{}) for the candidate numbering `mode` (0: exhaustive, 1: Philox)
template <class F>
static void with_mode(int mode, F&& f) {
  if (mode == 0) f(std::integral_constant<int, 0>{});
  else f(std::integral_constant<int, 1>{});
}

template <int M_, int K_, int N_, int RU_>
struct ShapeTag {
  static constexpr int M = M_, K = K_, N = N_;
  static constexpr int RU = RU_;  // > 0: orbit_sweep_kernel / orbit_sweep8_kernel with the row loop fully unrolled for r == RU
};

// The compiled shapes (m, k, n, unrolled r): calls f(ShapeTag<...>{}) for the first entry that matches -- r-specialised entries come
// first, the generic (RU = 0) entry of a shape last -- and returns false when none does.  f is instantiated for every entry, so the
// kernels that ignore RU instantiate once per (m, k, n).
template <class F>
static bool with_shape(int m, int k, int n, int r, F&& f) {
  bool hit = false;
  auto entry = [&](auto s) {
    using S = decltype(s);
    if (!hit && S::M == m && S::K == k && S::N == n && (S::RU == 0 || S::RU == r)) {
      hit = true;
      f(s);
    }
  };
  entry(ShapeTag<2, 2, 2, 7>{}); entry(ShapeTag<2, 2, 2, 0>{}); entry(ShapeTag<3, 3, 3, 0>{}); entry(ShapeTag<4, 4, 4, 0>{});
  entry(ShapeTag<3, 4, 7, 0>{}); entry(ShapeTag<3, 3, 6, 0>{}); entry(ShapeTag<3, 6, 3, 0>{}); entry(ShapeTag<6, 3, 3, 0>{});
  return hit;
}

// ---------------------------------------------------------------------------
// Runtime-shape kernels: (m, k, n) are kernel arguments, any dimension from 1 to kMaxDim, so every shape runs without being
// compiled in (rotations such as <4,7,3>, Kronecker products such as Strassen (x) <1,1,2>, naive <5,5,5>, ...).  One candidate
// per thread, as everywhere else: the reads of L | R | P^T from the constant bank stay warp-uniform.  The six factors U, U^-1,
// V, V^-1, W, W^-1 live as int8 in a thread-private column of shared memory (element e of thread t at byte e.kThreads + t: a
// warp reads 32 consecutive bytes, conflict-free); inverse entries of a zoi matrix are at most 2^(s-2) = 64 in magnitude.
// Arithmetic is int64 throughout: with int32 inputs every transformed entry is below 2^42, with int64 inputs below 2^46 it stays
// below 2^60 (host-checked).  Entries are classified as they come out of the second product stage; no transformed row is
// stored.  G2 follows the per-row order and rounding of the compiled kernels: `narrow` plans (the int32 magnitude bound holds)
// sum exact integer squares per row and scale once without contraction, like orbit_sweep_kernel (integer triples bit-exact
// against the reference formula, bit-identical to the compiled kernels); the others scale every entry first and use the two FMAs
// nvcc contracts in orbit_wide_kernel, within 1e-12 relative of the reference and within a few ulps of orbit_wide_kernel (counts
// and sparsity winners identical).  p != 0: Z/pZ sparsity.
// ---------------------------------------------------------------------------
struct RtArgs {
  int m, k, n, r, mode, measure;
  int narrow;          // 1: exact integer row sums of squares, G2 scaled by inv_prod at the end
  int g2;              // 1: evaluate G2 (growth-factor sweeps, tables, the winner's record)
  Den3 den;
  double3 inv_den;     // per-entry scale of the wide G2
  double inv_prod;     // 1 / (denL.denR.denP)
  ModP mp;             // mp.p != 0: residues, sparsity over Z/pZ
  unsigned long long seed;
};
// Quadratic plans: sqrt(d) of the real embedding (d > 0), with which G2 converts an entry (a + b.sqrt(d)) / den to a double.  It sits
// in the constant bank rather than in RtArgs, so that the rational instantiations keep their parameter layout.
__constant__ double c_sqrtd;

// Runtime-s twin of decode_zoi: the same digits in the same order (s = 1: one sign digit; a fresh word per matrix in Philox mode).
template <class DS>
__host__ __device__ __forceinline__ Zoi decode_zoi_rt(DS& ds, int s) {
  Zoi z;
  ds.start_matrix();
  z.pP = 0x76543210u;
  z.pQ = 0x76543210u;
  for (int i = 0; i + 1 < s; ++i) z.pP = nibble_swap(z.pP, i, ds.digit((uint32_t)(s - i)));
  for (int i = 0; i + 1 < s; ++i) z.pQ = nibble_swap(z.pQ, i, ds.digit((uint32_t)(s - i)));
  z.D = 0;
  for (int i = 0; i < s; ++i) z.D |= ds.digit(2u) << i;
  z.T = 0;
  for (int idx = 0; idx < s * (s - 1) / 2; ++idx) z.T |= (unsigned long long)ds.digit(3u) << (2 * idx);
  return z;
}

// M (s x s) and M^-1 as int8 with element stride `st` bytes (see expand_zoi for the layout).  T^-1 is built in M's slots first.
__host__ __device__ __forceinline__ void expand_zoi_rt(const Zoi& z, int s, signed char* M, signed char* Mi, int st) {
  auto t = [&](int i, int j) -> int {  // T[i][j], i <= j
    if (i == j) return ((z.D >> i) & 1u) ? 1 : -1;
    return (int)((z.T >> (2 * (i * s - i * (i + 1) / 2 + (j - i - 1)))) & 3ull) - 1;
  };
  for (int j = 0; j < s; ++j) {  // back substitution, as in expand_zoi
    M[(j * s + j) * st] = (signed char)t(j, j);
    for (int i = j - 1; i >= 0; --i) {
      int acc = 0;
      for (int q = i + 1; q <= j; ++q) acc += t(i, q) * M[(q * s + j) * st];
      M[(i * s + j) * st] = (signed char)(-t(i, i) * acc);
    }
  }
  for (int e = 0; e < s * s; ++e) Mi[e * st] = 0;
  for (int i = 0; i < s; ++i)
    for (int j = i; j < s; ++j) Mi[((int)((z.pQ >> (4 * i)) & 15u) * s + (int)((z.pP >> (4 * j)) & 15u)) * st] = M[(i * s + j) * st];
  for (int e = 0; e < s * s; ++e) M[e * st] = 0;
  for (int i = 0; i < s; ++i)
    for (int j = i; j < s; ++j) M[((int)((z.pP >> (4 * i)) & 15u) * s + (int)((z.pQ >> (4 * j)) & 15u)) * st] = (signed char)t(i, j);
}

struct AccRt {
  int nnz, nno;
  long long isq;  // narrow G2
  double sq;      // wide G2
};

__device__ __forceinline__ void classify_rt(long long s, long long den, double inv_den, const RtArgs& a, AccRt& acc) {
  if (a.mp.p) {
    const unsigned int v = modp_reduce(s, a.mp);
    acc.nnz += (v != 0u);
    acc.nno += (v != 0u) & (v != 1u) & (v != a.mp.p - 1u);
  } else {
    acc.nnz += (s != 0);
    acc.nno += (s != 0) & (s != den) & (s != -den);
    if (a.g2) {
      if (a.narrow) acc.isq += s * s;
      else {
        const double v = __dmul_rn((double)s, inv_den);
        acc.sq = __fma_rn(v, v, acc.sq);  // orbit_wide_kernel's `acc.sq += v * v`, contracted as nvcc contracts it there
      }
    }
  }
}

// The same over Q(sqrt d) for an entry (s + t.sqrt(d)) / den: zero iff both parts are, +-1 iff t = 0 and s = +-den; G2 squares the
// double value of the entry (growthfactor.cpp:25-28), so there is no exact-integer narrow form.
__device__ __forceinline__ void classify_pair_rt(long long s, long long t, long long den, double inv_den, const RtArgs& a, AccRt& acc) {
  const bool nz = (s | t) != 0;
  acc.nnz += nz;
  acc.nno += nz & !((t == 0) & ((s == den) | (s == -den)));
  if (a.g2) {
    const double v = __dmul_rn(__fma_rn((double)t, c_sqrtd, (double)s), inv_den);
    acc.sq = __fma_rn(v, v, acc.sq);
  }
}

// Y = Lm'.A.Rm' for one row A (ra x ca) with Lm'[x][i] = Lf[x.lsx + i.lsi], Rm'[j][y] = Rf[j.rsj + y.rsy]; every entry of Y is
// classified as it comes out.  The register-resident dimension of the intermediate is unrolled to kMaxDim with guards, which
// compile to predicated (not skipped) iterations, so it costs kMaxDim whatever its size: row by row (intermediate X = Lm'.A,
// kMaxDim.(ra.ra + ra.ca) multiply-adds) or column by column (Z = A.Rm', kMaxDim.(ca.ca + ra.ca)).  Taking the smaller square
// makes the work per candidate symmetric in (m, k, n) -- the three products cover every pair of dimensions once.  The wide G2
// sums squares in orbit_wide_kernel's row-major order, so it always goes row by row.
template <typename TA>
__device__ __forceinline__ void transform_row_rt(const TA* __restrict__ A, int ra, int ca, const signed char* Lf, int lsx, int lsi,
                                                 const signed char* Rf, int rsj, int rsy, long long den, double inv_den, const RtArgs& a,
                                                 AccRt& acc) {
  if (ca < ra && (a.narrow || !a.g2 || a.mp.p)) {
    for (int y = 0; y < ca; ++y) {
      long long Z[kMaxDim];
#pragma unroll
      for (int i = 0; i < kMaxDim; ++i) Z[i] = 0;
      for (int j = 0; j < ca; ++j) {
        const long long rv = Rf[j * rsj + y * rsy];
#pragma unroll
        for (int i = 0; i < kMaxDim; ++i)
          if (i < ra) Z[i] += (long long)A[i * ca + j] * rv;
      }
      for (int x = 0; x < ra; ++x) {
        long long v = 0;
#pragma unroll
        for (int i = 0; i < kMaxDim; ++i)
          if (i < ra) v += Z[i] * (long long)Lf[x * lsx + i * lsi];
        classify_rt(v, den, inv_den, a, acc);
      }
    }
    return;
  }
  for (int x = 0; x < ra; ++x) {
    long long X[kMaxDim];
#pragma unroll
    for (int j = 0; j < kMaxDim; ++j) X[j] = 0;
    for (int i = 0; i < ra; ++i) {
      const long long l = Lf[x * lsx + i * lsi];
      const TA* Ai = A + i * ca;
#pragma unroll
      for (int j = 0; j < kMaxDim; ++j)
        if (j < ca) X[j] += l * (long long)Ai[j];
    }
    for (int y = 0; y < ca; ++y) {
      long long v = 0;
#pragma unroll
      for (int j = 0; j < kMaxDim; ++j)
        if (j < ca) v += X[j] * (long long)Rf[j * rsj + y * rsy];
      classify_rt(v, den, inv_den, a, acc);
    }
  }
}

// transform_row_rt over Q(sqrt d): the rows A and B of both parts go through every factor entry read once, row by row (the order
// of the wide G2), and each entry (A' + B'.sqrt(d)) / den is classified as a pair.
template <typename TA>
__device__ __forceinline__ void transform_pair_rt(const TA* __restrict__ A, const TA* __restrict__ B, int ra, int ca, const signed char* Lf, int lsx,
                                                  int lsi, const signed char* Rf, int rsj, int rsy, long long den, double inv_den, const RtArgs& a,
                                                  AccRt& acc) {
  for (int x = 0; x < ra; ++x) {
    long long X[kMaxDim], Xb[kMaxDim];
#pragma unroll
    for (int j = 0; j < kMaxDim; ++j) X[j] = Xb[j] = 0;
    for (int i = 0; i < ra; ++i) {
      const long long l = Lf[x * lsx + i * lsi];
      const TA* Ai = A + i * ca;
      const TA* Bi = B + i * ca;
#pragma unroll
      for (int j = 0; j < kMaxDim; ++j)
        if (j < ca) {
          X[j] += l * (long long)Ai[j];
          Xb[j] += l * (long long)Bi[j];
        }
    }
    for (int y = 0; y < ca; ++y) {
      long long v = 0, vb = 0;
#pragma unroll
      for (int j = 0; j < kMaxDim; ++j)
        if (j < ca) {
          const long long rv = Rf[j * rsj + y * rsy];
          v += X[j] * rv;
          vb += Xb[j] * rv;
        }
      classify_pair_rt(v, vb, den, inv_den, a, acc);
    }
  }
}

// Scores one candidate; f = this thread's column of the factor scratch.  Unscaled G2 for narrow plans (the sweep's key).  Q: entries
// in Q(sqrt d).
template <typename TA, int MODE, bool Q = false>
__device__ __forceinline__ Score score_candidate_rt(const TA* __restrict__ lrp, const RtArgs& a, unsigned long long index, signed char* f) {
  constexpr int st = kThreads;
  const int m = a.m, k = a.k, n = a.n;
  signed char *U = f, *Ui = U + m * m * st, *V = Ui + m * m * st, *Vi = V + k * k * st, *W = Vi + k * k * st, *Wi = W + n * n * st;
  Digits<MODE> ds(a.seed, index);
  {
    const Zoi z = decode_zoi_rt(ds, m);
    expand_zoi_rt(z, m, U, Ui, st);
  }
  {
    const Zoi z = decode_zoi_rt(ds, k);
    expand_zoi_rt(z, k, V, Vi, st);
  }
  {
    const Zoi z = decode_zoi_rt(ds, n);
    expand_zoi_rt(z, n, W, Wi, st);
  }
  const TA* Lc = lrp;
  const TA* Rc = Lc + a.r * m * k;
  const TA* Pc = Rc + a.r * k * n;
  Score sc;
  sc.nnz = 0; sc.nno = 0; sc.g2 = 0.0;
  for (int l = 0; l < a.r; ++l) {
    AccRt aL, aR, aP;
    aL.nnz = aL.nno = 0; aL.isq = 0; aL.sq = 0.0;
    aR = aL; aP = aL;
    if constexpr (Q) {  // the sqrt(d) parts of L | R | P^T follow the rational parts in the constant bank, in the same layout
      const int part = a.r * (m * k + k * n + m * n);
      transform_pair_rt<TA>(Lc + l * m * k, Lc + l * m * k + part, m, k, Ui, st, m * st, V, k * st, st, a.den.x, a.inv_den.x, a, aL);
      transform_pair_rt<TA>(Rc + l * k * n, Rc + l * k * n + part, k, n, Vi, k * st, st, W, n * st, st, a.den.y, a.inv_den.y, a, aR);
      transform_pair_rt<TA>(Pc + l * m * n, Pc + l * m * n + part, m, n, U, m * st, st, Wi, st, n * st, a.den.z, a.inv_den.z, a, aP);
    } else {
      transform_row_rt<TA>(Lc + l * m * k, m, k, Ui, st, m * st, V, k * st, st, a.den.x, a.inv_den.x, a, aL);   // U^-T A V
      transform_row_rt<TA>(Rc + l * k * n, k, n, Vi, k * st, st, W, n * st, st, a.den.y, a.inv_den.y, a, aR);   // V^-1 B W
      transform_row_rt<TA>(Pc + l * m * n, m, n, U, m * st, st, Wi, st, n * st, a.den.z, a.inv_den.z, a, aP);   // U C W^-T
    }
    sc.nnz += (uint32_t)(aL.nnz + aR.nnz + aP.nnz);
    sc.nno += (uint32_t)(aL.nno + aR.nno + aP.nno);
    if (a.g2) {  // growthfactor.cpp:117-125, rows in order, each path rounded exactly as its compiled counterpart
      if (a.narrow)  // orbit_sweep_kernel / orbit_table_kernel: no contraction
        sc.g2 = __dadd_rn(sc.g2, __dmul_rn(__dmul_rn(sqrt((double)aL.isq), sqrt((double)aR.isq)), sqrt((double)aP.isq)));
      else  // orbit_wide_kernel: `sc.g2 += (a * b) * c`, the outer product and the sum contracted
        sc.g2 = __fma_rn(__dmul_rn(sqrt(aL.sq), sqrt(aR.sq)), sqrt(aP.sq), sc.g2);
    }
  }
  return sc;
}

__device__ __forceinline__ double rt_score_g2(const RtArgs& a, const Score& s) { return a.narrow ? s.g2 * a.inv_prod : s.g2; }

// Grid-stride over [lo,hi) in whole warps (sink_emit is warp-collective); per-block best to block_best, optional tables and sink.
// Q: the entries lie in Q(sqrt d) (plo_orbit_plan_create_quad).
template <typename TA, int MODE, bool Q = false>
__global__ void __launch_bounds__(kThreads) orbit_rt_kernel(RtArgs a, unsigned long long lo, unsigned long long hi, Key* __restrict__ block_best,
                                                             uint32_t* __restrict__ tnnz, uint32_t* __restrict__ tnno, double* __restrict__ tg2,
                                                             Sink sink) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ Key red[32];
  signed char* f = reinterpret_cast<signed char*>(dyn_smem) + threadIdx.x;
  const TA* lrp = reinterpret_cast<const TA*>(c_lrp);
  const unsigned long long stride = (unsigned long long)gridDim.x * kThreads;
  const int lane = threadIdx.x & 31;
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (unsigned long long wb = lo + (unsigned long long)blockIdx.x * kThreads + (threadIdx.x - lane); wb < hi; wb += stride) {
    const unsigned long long idx = wb + lane;
    const bool valid = idx < hi;
    Score s;
    s.nnz = 0; s.nno = 0; s.g2 = 0.0;
    double g2 = 0.0;
    if (valid) {
      s = score_candidate_rt<TA, MODE, Q>(lrp, a, idx, f);
      g2 = rt_score_g2(a, s);
      if (tnnz) tnnz[idx - lo] = s.nnz;
      if (tnno) tnno[idx - lo] = s.nno;
      if (tg2) tg2[idx - lo] = g2;
      Key k;
      k.primary = a.measure == PLO_MEASURE_G2 ? (unsigned long long)__double_as_longlong(s.g2) : (((unsigned long long)s.nnz << 32) | s.nno);
      k.index = idx;
      if (k.primary < best.primary) best = k;
    }
    if (sink.rec) sink_emit(sink, valid, idx, s.nnz, s.nno, g2);
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) block_best[blockIdx.x] = best;
}

// Reduces the per-block keys and writes the winner's record with both measures (the plan's device result: plo_orbit_plan_pack).
template <typename TA, int MODE, bool Q = false>
__global__ void __launch_bounds__(kThreads) orbit_rt_final_kernel(RtArgs a, int nblocks, const Key* __restrict__ block_best,
                                                                   plo_orbit_best* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ Key red[32];
  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  for (int b = threadIdx.x; b < nblocks; b += kThreads) {
    const Key k = block_best[b];
    if (key_less(k, best)) best = k;
  }
  best = block_min(best, red);
  if (threadIdx.x == 0) {
    plo_orbit_best o;
    o.index = best.index;
    o.nnz = 0; o.nno = 0; o.score = 0.0;
    if (best.index != ~0ull) {
      RtArgs b = a;
      b.g2 = a.mp.p == 0u;
      const Score s = score_candidate_rt<TA, MODE, Q>(reinterpret_cast<const TA*>(c_lrp), b, best.index, reinterpret_cast<signed char*>(dyn_smem));
      o.nnz = s.nnz; o.nno = s.nno;
      o.score = (a.measure == PLO_MEASURE_G2 && a.mp.p == 0u) ? rt_score_g2(b, s) : (double)s.nnz;
    }
    *out = o;
  }
}

static size_t rt_smem(int m, int k, int n) { return (size_t)2 * (m * m + k * k + n * n) * kThreads; }

template <typename TA, bool Q = false>
static void rt_launch(const RtArgs& a, int grid, cudaStream_t st, unsigned long long lo, unsigned long long hi, Key* bb, uint32_t* tnnz,
                      uint32_t* tnno, double* tg2, Sink sink) {
  const size_t smem = rt_smem(a.m, a.k, a.n);
  with_mode(a.mode, [&](auto md) { orbit_rt_kernel<TA, decltype(md)::value, Q><<<grid, kThreads, smem, st>>>(a, lo, hi, bb, tnnz, tnno, tg2, sink); });
}
template <typename TA, bool Q = false>
static void rt_final(const RtArgs& a, int nblocks, cudaStream_t st, const Key* bb, plo_orbit_best* out) {
  const size_t smem = rt_smem(a.m, a.k, a.n);
  with_mode(a.mode, [&](auto md) { orbit_rt_final_kernel<TA, decltype(md)::value, Q><<<1, kThreads, smem, st>>>(a, nblocks, bb, out); });
}
// Opts the kernels in to the factor scratch of the largest shape (the attribute belongs to the function, which every live
// runtime-shape plan shares: lowering it for a small shape would break the launches of a larger plan); returns blocks per SM for
// this shape (0: cannot run, error message set).
template <typename TA, bool Q = false>
static int rt_prepare(int m, int k, int n) {
  const int most = (int)rt_smem(kMaxDim, kMaxDim, kMaxDim);
  int nb = 0;
  if (cudaFuncSetAttribute(orbit_rt_kernel<TA, 0, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, most) != cudaSuccess ||
      cudaFuncSetAttribute(orbit_rt_kernel<TA, 1, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, most) != cudaSuccess ||
      cudaFuncSetAttribute(orbit_rt_final_kernel<TA, 0, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, most) != cudaSuccess ||
      cudaFuncSetAttribute(orbit_rt_final_kernel<TA, 1, Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, most) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, orbit_rt_kernel<TA, 1, Q>, kThreads, rt_smem(m, k, n)) != cudaSuccess || nb < 1) {
    cudaGetLastError();
    set_error("orbit sweep: cannot reserve %zu bytes of shared memory for the runtime-shape kernel", rt_smem(m, k, n));
    return 0;
  }
  return nb;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
using SweepKernel = void (*)(int, int3, unsigned long long, unsigned long long, unsigned long long, int, Key*);

// The orbit_sweep_kernel variant for a measure, a sqrt table that covers every row norm^2 (lutfull) and two 16-bit lanes (pack)
template <class S, int MODE>
static SweepKernel sweep_kernel(int measure, bool lutfull, bool pack) {
  constexpr int M = S::M, K = S::K, N = S::N, RU = S::RU;
  if (measure == PLO_MEASURE_NNZ)
    return pack ? &orbit_sweep_kernel<M, K, N, MODE, PLO_MEASURE_NNZ, RU, false, true> : &orbit_sweep_kernel<M, K, N, MODE, PLO_MEASURE_NNZ, RU, false, false>;
  if (lutfull) return pack ? &orbit_sweep_kernel<M, K, N, MODE, PLO_MEASURE_G2, RU, true, true> : &orbit_sweep_kernel<M, K, N, MODE, PLO_MEASURE_G2, RU, true, false>;
  return pack ? &orbit_sweep_kernel<M, K, N, MODE, PLO_MEASURE_G2, RU, false, true> : &orbit_sweep_kernel<M, K, N, MODE, PLO_MEASURE_G2, RU, false, false>;
}

// Lets kernel f use `smem` bytes of dynamic shared memory; false (error cleared) when the device refuses.
template <class F>
static bool allow_smem(F f, size_t smem) {
  if (cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess) return true;
  cudaGetLastError();
  return false;
}
// Resident blocks per SM of kernel f with `threads` threads and `smem` bytes of dynamic shared memory (0: cannot run).
template <class F>
static int blocks_per_sm(F f, int threads, size_t smem) {
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, f, threads, smem) == cudaSuccess) return nb;
  cudaGetLastError();
  return 0;
}
// The same for a kernel whose two modes (f0, f1) may need more than the default 48 KB: both are opted in first.
template <class F>
static int blocks_per_sm(F f0, F f1, int threads, size_t smem) {
  if (smem > 48 * 1024 && !(allow_smem(f0, smem) && allow_smem(f1, smem))) return 0;
  return blocks_per_sm(f1, threads, smem);
}

// Worst-case magnitude bound of the transformed entries (host guard for the int32 arithmetic and for the lane packings).
// Only the FINAL entries matter: the packed multiply-adds are plain arithmetic modulo 2^32, so an intermediate lane may spill as
// long as every final lane is inside its range.  A row (or column) of the inverse of a zoi matrix is a permuted row of T^-1 with
// |T^-1[i][j]| <= 2^(j-i-1) (j > i), 1 on the diagonal, so its magnitudes sorted in decreasing order are dominated by
// g(s) = (2^(s-2), .., 2, 1, 1); the {-1,0,1} factor on the other side contributes at most 1 per term.  Hence, per row l,
//   |U^-T A_l V| <= sum_t g(m)_t . (row sums of |A_l|, decreasing)_t      (rearrangement inequality)
//   |V^-1 B_l W| <= sum_t g(k)_t . (row sums of |B_l|, decreasing)_t
//   |U C_l W^-T| <= sum_t g(n)_t . (column sums of |C_l|, decreasing)_t
// which follows the actual sparsity of the Hopcroft-Musinski rows instead of max|entry| . 2^(s-1) . dimension
// (3x4x7_63_rational: 6 / 56 / 96 instead of 16 / 112 / 192, which admits the four-lane kernels).
template <typename T>
static long long tight_bound(const T* A, int r, int ra, int ca, size_t row_stride, size_t elt_stride, bool by_rows) {
  const int s = by_rows ? ra : ca, other = by_rows ? ca : ra;
  long long g[kMaxDim], sums[kMaxDim], worst = 0;
  g[0] = 1;
  for (int t = 1; t < s; ++t) g[t] = 1ll << (t - 1);
  std::sort(g, g + s, [](long long a, long long b) { return a > b; });
  for (int l = 0; l < r; ++l) {
    for (int t = 0; t < s; ++t) {
      long long acc = 0;
      for (int o = 0; o < other; ++o) {
        const int i = by_rows ? t : o, j = by_rows ? o : t;
        const long long v = A[(size_t)l * row_stride + (size_t)(i * ca + j) * elt_stride];
        acc += v < 0 ? -v : v;
      }
      sums[t] = acc;
    }
    std::sort(sums, sums + s, [](long long a, long long b) { return a > b; });
    long long b = 0;
    for (int t = 0; t < s; ++t) b += g[t] * sums[t];
    if (b > worst) worst = b;
  }
  return worst;
}

static bool magnitude_ok(int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, long long* smax, bool* lanes16, bool* lanes8 = nullptr,
                         long long* bounds = nullptr) {
  if (m > kMaxDim || k > kMaxDim || n > kMaxDim) return false;
  const long long bl = tight_bound(L, r, m, k, (size_t)m * k, 1, true);   // L: r x (m*k), row l = vec(A_l)
  const long long br = tight_bound(R, r, k, n, (size_t)k * n, 1, true);   // R: r x (k*n)
  const long long bp = tight_bound(P, r, m, n, 1, (size_t)r, false);      // P: (m*n) x r, column l = vec(C_l)
  if (bounds) { bounds[0] = bl; bounds[1] = br; bounds[2] = bp; }
  auto ok = [](long long b, int cnt) { return b < 46340 && b * b * cnt < 2147483647ll; };
  if (!(ok(bl, m * k) && ok(br, k * n) && ok(bp, m * n))) return false;
  long long s = bl * bl * m * k;
  if (br * br * k * n > s) s = br * br * k * n;
  if (bp * bp * m * n > s) s = bp * bp * m * n;
  *smax = s;
  *lanes16 = bl < 32768 && br < 32768 && bp < 32768;  // two-lane packing stays exact
  if (lanes8) *lanes8 = bl < 128 && br < 128 && bp < 128;  // four-lane packing stays exact
  return true;
}

// Runtime-shape dispatch.  plo_set_orbit_any_shape(1) sends the shapes that have no compiled kernel to the runtime-shape kernels;
// PLO_ORBIT_RUNTIME_SHAPE in the environment sends the compiled shapes there too (A/B timing and parity: same results, G2 of the 64-bit paths up to the last bits).
static int g_any_shape = 0;
// *rt = the shape runs on the runtime-shape kernels, else on its compiled ones; PLO_E_SHAPE when it has neither.
static int orbit_route(int m, int k, int n, int r, bool* rt) {
  const bool compiled = with_shape(m, k, n, r, [](auto) {});
  *rt = compiled ? getenv("PLO_ORBIT_RUNTIME_SHAPE") != nullptr : g_any_shape != 0;
  if (compiled || *rt) return PLO_OK;
  set_error("orbit sweep: shape %dx%dx%d not compiled in", m, k, n);
  return PLO_E_SHAPE;
}

// Limits of every orbit sweep; `words` = constant-bank ints per entry (2 for int64 inputs)
static int orbit_limits(int m, int k, int n, int r, int mode, int words) {
  if (m < 1 || k < 1 || n < 1 || m > kMaxDim || k > kMaxDim || n > kMaxDim) {
    set_error("orbit sweep: %dx%dx%d: dimensions must be between 1 and %d (nibble-packed permutations)", m, k, n, kMaxDim);
    return PLO_E_SHAPE;
  }
  const long long ints = (long long)words * r * (m * k + k * n + m * n);
  if (ints > kConstInts) {
    set_error("orbit sweep: L/R/P of %dx%dx%d, r = %d need %lld constant-bank ints, the bank holds %d", m, k, n, r, ints, kConstInts);
    return PLO_E_SHAPE;
  }
  if (mode == 0 && plo_orbit_space(m, k, n) == 0) { set_error("orbit sweep: exhaustive space of %dx%dx%d exceeds 64 bits", m, k, n); return PLO_E_SHAPE; }
  return PLO_OK;
}
// every transformed entry below 2^62 (int64 arithmetic of the runtime-shape kernels)
template <typename T>
static bool rt_bound_ok(int m, int k, int n, int r, const T* L, const T* R, const T* P) {
  const long long lim = 1ll << 62;
  return tight_bound(L, r, m, k, (size_t)m * k, 1, true) < lim && tight_bound(R, r, k, n, (size_t)k * n, 1, true) < lim &&
         tight_bound(P, r, m, n, 1, (size_t)r, false) < lim;
}
static Den3 abs_den(long long a, long long b, long long c) { return Den3{a < 0 ? -a : a, b < 0 ? -b : b, c < 0 ? -c : c}; }
static double3 inverses(Den3 d) { return make_double3(1.0 / (double)d.x, 1.0 / (double)d.y, 1.0 / (double)d.z); }
static ModP make_modp(uint32_t p) {
  ModP mp;
  mp.p = p; mp.M64 = 0; mp.bias = 0;
  if (p) { mp.M64 = ~0ull / p; mp.bias = (((1ull << 48) + p - 1) / p) * p; }  // |entry| < 2^43 over Z/pZ
  return mp;
}
static RtArgs rt_args(int m, int k, int n, int r, int mode, int measure, uint64_t seed, Den3 den, bool narrow, uint32_t p) {
  RtArgs a;
  a.m = m; a.k = k; a.n = n; a.r = r; a.mode = mode; a.measure = measure; a.seed = seed;
  a.narrow = narrow ? 1 : 0;
  a.g2 = measure == PLO_MEASURE_G2 && p == 0;
  a.den = den;
  a.inv_den = inverses(den);
  a.inv_prod = 1.0 / ((double)den.x * (double)den.y * (double)den.z);
  a.mp = make_modp(p);
  return a;
}

// which plan's L/R/P currently sits in the constant bank of each device (constant memory is per device)
constexpr int kMaxDevices = 64;
static const void* g_const_owner_dev[kMaxDevices] = {nullptr};
static const void*& const_owner() {
  int d = 0;
  cudaGetDevice(&d);
  return g_const_owner_dev[(d >= 0 && d < kMaxDevices) ? d : 0];
}
// The constant bank is shared by every plan of a device, and plan_run is asynchronous: before the bank is re-written, or read from
// another stream than the one that wrote it, that stream waits for an event recorded after the bank's last use.  This makes one host
// thread driving several streams (or alternating plans) safe; two host threads on one device are still excluded (plinopt_b200.h).
static cudaEvent_t g_bank_event[kMaxDevices] = {nullptr};
static cudaStream_t g_bank_stream[kMaxDevices] = {nullptr};
static bool g_bank_used[kMaxDevices] = {false};
static int bank_device() {
  int d = 0;
  cudaGetDevice(&d);
  return (d >= 0 && d < kMaxDevices) ? d : 0;
}
// call before uploading to the bank or launching a kernel that reads it on stream `st`
static void bank_acquire(cudaStream_t st, bool rewriting) {
  const int d = bank_device();
  if (g_bank_used[d] && g_bank_event[d] && (rewriting || g_bank_stream[d] != st)) cudaStreamWaitEvent(st, g_bank_event[d], 0);
}
// call after the last launch of a sequence that reads the bank on stream `st`
static void bank_release(cudaStream_t st) {
  const int d = bank_device();
  if (!g_bank_event[d] && cudaEventCreateWithFlags(&g_bank_event[d], cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); g_bank_event[d] = nullptr; return; }
  cudaEventRecord(g_bank_event[d], st);
  g_bank_stream[d] = st;
  g_bank_used[d] = true;
}

// Host-only self-test of the "whole matrix from one number" decode the table-driven kernels rely on (no device needed): for S = 2
// (48 matrices) and S = 3 (7776), drawing the digits of a matrix one by one from a word x gives the same matrix as replaying matrix
// number floor(x . count / 2^32) (Philox mode) resp. rem mod count (exhaustive mode).  Returns the number of mismatches.
template <int S, int COUNT>
static int matrix_index_mismatches() {
  int bad = 0;
  auto same = [](const Zoi& a, const Zoi& b) { return a.pP == b.pP && a.pQ == b.pQ && a.D == b.D && a.T == b.T; };
  for (uint32_t e = 0; e < (uint32_t)COUNT; ++e) {
    // the first, the last and a middle word of the slice of 2^32 that maps to e
    const uint32_t x0 = (uint32_t)((((unsigned long long)e << 32) + COUNT - 1) / COUNT);
    const uint32_t x1 = (uint32_t)(((((unsigned long long)e + 1) << 32) + COUNT - 1) / COUNT - 1);
    const uint32_t xs[3] = {x0, x1, x0 + (x1 - x0) / 2};
    RawDigits<1> ref(e, COUNT);
    const Zoi zr = decode_zoi<S, 1, RawDigits<1>>(ref);
    for (uint32_t x : xs) {
      if ((uint32_t)(((unsigned long long)x * COUNT) >> 32) != e) { ++bad; continue; }
      RawDigits<1> d(0, COUNT);
      d.x = x;
      if (!same(decode_zoi<S, 1, RawDigits<1>>(d), zr)) ++bad;
    }
    RawDigits<0> ref0(e, COUNT);
    const Zoi z0 = decode_zoi<S, 0, RawDigits<0>>(ref0);
    RawDigits<0> d0(0, COUNT);
    d0.rem = (unsigned long long)e + 5ull * COUNT;  // a larger running remainder: only rem mod count may matter
    if (!same(decode_zoi<S, 0, RawDigits<0>>(d0), z0)) ++bad;
  }
  return bad;
}
// Q(sqrt d) needs d not a perfect square (else X^2 - d is not irreducible); G2 needs the real embedding sqrt(d) > 0.  Shared with
// plo_growth_factors_quad (host_api.cpp).
int quad_field_ok(int64_t d, int measure, const char* who) {
  const long long rt = d >= 0 ? (long long)std::llround(std::sqrt((double)d)) : -1;
  bool square = false;
  for (long long t = rt - 1; t <= rt + 1 && !square; ++t) square = t >= 0 && t <= 3037000499ll && t * t == d;
  if (square) { set_error("%s: X^2 - %lld: d is a perfect square, Q(sqrt d) is not a field", who, (long long)d); return PLO_E_ARG; }
  if (measure == PLO_MEASURE_G2 && d < 0) { set_error("%s: G2 needs a real embedding of Q(sqrt %lld), d > 0", who, (long long)d); return PLO_E_ARG; }
  return PLO_OK;
}
}  // namespace plo

using namespace plo;

// The sweep kernel of a plan, chosen once when the plan is created.
enum class OrbitPath {
  Runtime,      // orbit_rt_kernel: any shape up to 8x8x8 (plo_set_orbit_any_shape, PLO_ORBIT_RUNTIME_SHAPE)
  Quadratic,    // orbit_rt_kernel<TA, MODE, true>: entries in Q(sqrt d), every shape up to 8x8x8 (plo_orbit_plan_create_quad)
  Wide,         // orbit_wide_kernel: exact 64-bit products (int32 product bound exceeded); winner picked on the host
  Table8x,      // orbit_sweep8x_kernel: 2x2x2, r = 7, growth factor, row measures per factor class pair from shared-memory tables
  Table2x,      // orbit_sweep2x_kernel: its sparsity twin
  FourLaneNnz,  // orbit_sweepn8_kernel: sparsity, transformed entries and denominators below 128
  FourLaneG2,   // orbit_sweep8_kernel: growth factor, transformed entries below 128
  Plain,        // orbit_sweep_kernel: one or two (pack) lanes
};

struct plo_orbit_plan {
  int m, k, n, r, measure, mode;
  unsigned long long seed;
  OrbitPath path;
  int3 den;              // |denominators|
  double inv_den;        // 1 / (denL.denR.denP)
  double3 inv_den3;      // 1 / |den| per factor (Wide)
  std::vector<int> h_lrp;
  std::vector<int> h_lrp2;  // c_lrp2: pairs of rows packed at 8-bit spacing (four-lane plans only)
  uint32_t h_pkeys[20];  // Philox round keys of `seed`
  int grid, lutn;        // blocks of the sweep kernel; sqrt table entries (growth factor)
  bool lutfull, pack;    // the sqrt table covers every row norm^2; Plain: two 16-bit lanes
  size_t smem;           // dynamic shared memory of the sweep kernel
  Key* d_block_best;
  plo_orbit_best* d_out;
  int4* d_z3tab;         // 3x3x3 four-lane plans: the 7776 zoi matrices of a factor, ready to use (1.5 MB, L2-resident)
  uint32_t* d_wide_cnt;  // Wide: [2] nnz, nno of the winner
  double* d_wide_g2;
  RtArgs rta;            // Runtime, Quadratic
  bool q64;              // Quadratic: the constant bank holds int64 entries
  double sqrtd;          // Quadratic: c_sqrtd (0 for d < 0: no G2)
};

// L | R | P^T (P^T row l = column l of P) as the constant bank holds them
template <typename T, typename S>
static void pack_lrp(std::vector<T>& h, int m, int k, int n, int r, const S* L, const S* R, const S* P) {
  h.resize((size_t)r * (m * k + k * n + m * n));
  T* dst = h.data();
  for (int i = 0; i < r * m * k; ++i) *dst++ = L[i];
  for (int i = 0; i < r * k * n; ++i) *dst++ = R[i];
  for (int l = 0; l < r; ++l)
    for (int e = 0; e < m * n; ++e) *dst++ = P[(size_t)e * r + l];
}

static Key min_key(const std::vector<Key>& bb) {
  Key b = bb[0];
  for (const Key& x : bb) if (key_less(x, b)) b = x;
  return b;
}

// f(ShapeTag, integral_constant MODE) for a plan of a compiled shape
template <class F>
static void with_plan(const plo_orbit_plan* pl, F&& f) {
  with_shape(pl->m, pl->k, pl->n, pl->r, [&](auto s) { with_mode(pl->mode, [&](auto md) { f(s, md); }); });
}

// f(TA{}, std::integral_constant<bool, Q>{}) for the runtime-shape kernel of a Runtime or Quadratic plan
template <class F>
static void with_rt(const plo_orbit_plan* pl, F&& f) {
  if (pl->path == OrbitPath::Runtime) f(int{}, std::false_type{});
  else if (pl->q64) f((long long){}, std::true_type{});
  else f(int{}, std::true_type{});
}

static void wide_launch(const plo_orbit_plan* pl, int grid, cudaStream_t st, uint64_t lo, uint64_t hi, Key* bb, uint32_t* tnnz, uint32_t* tnno,
                        double* tg2, Sink sink) {
  with_plan(pl, [&](auto s, auto md) {
    using S = decltype(s);
    orbit_wide_kernel<int, S::M, S::K, S::N, decltype(md)::value><<<grid, kThreads, 0, st>>>(pl->r, Den3{pl->den.x, pl->den.y, pl->den.z}, pl->inv_den3,
                                                                                             pl->measure, pl->seed, lo, hi, bb, tnnz, tnno, tg2, sink);
  });
}

// Synchronous sweep of [lo,hi) for the Z/pZ and 64-bit entry points: L | R | P^T (int32 or int64 words) into the constant bank,
// launch(grid, lo, hi, block_best, nnz, nno, g2) on the default stream with at most blocks_per_sm blocks per SM, the requested
// per-candidate tables back, the winner = the minimum of the block keys.  A sparsity key holds the winner's counts; for the growth
// factor one more launch on the winner alone returns all its measures.
template <typename TA, class Launch>
static int sweep_sync(const std::vector<TA>& h, int blocks_per_sm, int measure, uint64_t lo, uint64_t hi, Launch launch,
                      plo_orbit_best* best, uint32_t* tnnz, uint32_t* tnno, double* tg2) {
  const uint64_t cnt = hi - lo;
  const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((cnt + kThreads - 1) / kThreads, (uint64_t)sm_count() * blocks_per_sm));
  const bool rescore = best && measure == PLO_MEASURE_G2;
  Key* d_bb = nullptr;
  uint32_t *d_nnz = nullptr, *d_nno = nullptr, *d_one = nullptr;  // d_one: nnz, nno, g2 of the winner
  double* d_g2 = nullptr;
  const_owner() = nullptr;
  bank_acquire(nullptr, true);
  cudaError_t e = cudaMemcpyToSymbol(c_lrp, h.data(), h.size() * sizeof(TA));
  if (e == cudaSuccess) e = pool_alloc(&d_bb, sizeof(Key) * grid);
  if (e == cudaSuccess && tnnz && cnt) e = pool_alloc(&d_nnz, cnt * 4);
  if (e == cudaSuccess && tnno && cnt) e = pool_alloc(&d_nno, cnt * 4);
  if (e == cudaSuccess && tg2 && cnt) e = pool_alloc(&d_g2, cnt * 8);
  if (e == cudaSuccess && rescore) e = pool_alloc(&d_one, 16);
  if (e == cudaSuccess) {
    launch(grid, lo, hi, d_bb, d_nnz, d_nno, d_g2);
    e = cudaGetLastError();
  }
  std::vector<Key> bb((size_t)grid);
  if (e == cudaSuccess) e = cudaMemcpy(bb.data(), d_bb, sizeof(Key) * grid, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && d_nnz) e = cudaMemcpy(tnnz, d_nnz, cnt * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && d_nno) e = cudaMemcpy(tnno, d_nno, cnt * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && d_g2) e = cudaMemcpy(tg2, d_g2, cnt * 8, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && best) {
    const Key b = min_key(bb);
    best->index = b.index; best->nnz = 0; best->nno = 0; best->score = 0.0;
    if (b.index != ~0ull && !rescore) {
      best->nnz = (uint32_t)(b.primary >> 32); best->nno = (uint32_t)b.primary; best->score = (double)best->nnz;
    } else if (b.index != ~0ull) {
      launch(1, b.index, b.index + 1, d_bb, d_one, d_one + 1, reinterpret_cast<double*>(d_one + 2));
      uint32_t one[4];
      e = cudaMemcpy(one, d_one, 16, cudaMemcpyDeviceToHost);
      best->nnz = one[0]; best->nno = one[1];
      std::memcpy(&best->score, one + 2, 8);
    }
  }
  pool_free(d_bb); pool_free(d_nnz); pool_free(d_nno); pool_free(d_g2); pool_free(d_one);
  if (e != cudaSuccess) { set_error("orbit sweep: %s", cudaGetErrorString(e)); return PLO_E_CUDA; }
  return PLO_OK;
}

// sweep_sync on the runtime-shape kernel
template <typename TA>
static int rt_sync(const RtArgs& a, const std::vector<TA>& h, uint64_t lo, uint64_t hi, plo_orbit_best* best, uint32_t* tnnz, uint32_t* tnno, double* tg2) {
  const int nb = rt_prepare<TA>(a.m, a.k, a.n);
  if (nb < 1) return PLO_E_CUDA;
  return sweep_sync(h, nb, a.measure, lo, hi, [&](int grid, uint64_t l, uint64_t u, Key* bb, uint32_t* c0, uint32_t* c1, double* g) {
    rt_launch<TA>(a, grid, nullptr, l, u, bb, c0, c1, g, no_sink());
  }, best, tnnz, tnno, tg2);
}

// Z/pZ sweep: residues in, winner (and optional per-candidate table) out.  Synchronous.
static int orbit_modp(uint32_t p, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int mode, uint64_t seed,
                      uint64_t lo, uint64_t hi, plo_orbit_best* best, uint32_t* tnnz, uint32_t* tnno) {
  if (!L || !R || !P || r < 1 || p < 2 || p >= (1u << 31) || (mode != 0 && mode != 1) || hi < lo) {
    set_error("orbit sweep mod p: bad argument (need 2 <= p < 2^31)");
    return PLO_E_ARG;
  }
  int rc = check_device();
  if (rc) return rc;
  bool rt = false;
  if ((rc = orbit_route(m, k, n, r, &rt)) || (rc = orbit_limits(m, k, n, r, mode, 1))) return rc;
  auto residues = [p](const int32_t* A, size_t cnt) { return std::all_of(A, A + cnt, [p](int32_t v) { return v >= 0 && (uint32_t)v < p; }); };
  if (!residues(L, (size_t)r * m * k) || !residues(R, (size_t)r * k * n) || !residues(P, (size_t)r * m * n)) {
    set_error("orbit sweep mod p: residue out of range");
    return PLO_E_ARG;
  }
  std::vector<int> h;
  pack_lrp(h, m, k, n, r, L, R, P);
  if (rt) return rt_sync<int>(rt_args(m, k, n, r, mode, PLO_MEASURE_NNZ, seed, Den3{1, 1, 1}, false, p), h, lo, hi, best, tnnz, tnno, nullptr);
  const ModP mp = make_modp(p);
  with_shape(m, k, n, r, [&](auto s) {
    using S = decltype(s);
    rc = sweep_sync(h, 4, PLO_MEASURE_NNZ, lo, hi, [&](int grid, uint64_t l, uint64_t u, Key* bb, uint32_t* c0, uint32_t* c1, double*) {
      with_mode(mode, [&](auto md) { orbit_modp_kernel<S::M, S::K, S::N, decltype(md)::value><<<grid, kThreads>>>(r, mp, seed, l, u, bb, c0, c1); });
    }, best, tnnz, tnno, nullptr);
  });
  return rc;
}

// 64-bit inputs (common denominators beyond 2^31, e.g. 2x2x2_7_DPS-intermediate-12.0695): same exact 64-bit kernels, the constant
// bank holds int64 entries.  |entries| < 2^46 keeps both product stages inside 64 bits.  Synchronous; winner and/or per-candidate table.
static int orbit_wide64(int m, int k, int n, int r, const int64_t* L, const int64_t* R, const int64_t* P, int64_t denL, int64_t denR, int64_t denP,
                        int measure, int mode, uint64_t seed, uint64_t lo, uint64_t hi, plo_orbit_best* best, uint32_t* tnnz, uint32_t* tnno, double* tg2) {
  if (!L || !R || !P || r < 1 || denL == 0 || denR == 0 || denP == 0 || (measure != PLO_MEASURE_NNZ && measure != PLO_MEASURE_G2) ||
      (mode != 0 && mode != 1) || hi < lo) { set_error("orbit sweep (64-bit inputs): bad argument"); return PLO_E_ARG; }
  int rc = check_device();
  if (rc) return rc;
  bool rt = false;
  if ((rc = orbit_route(m, k, n, r, &rt)) || (rc = orbit_limits(m, k, n, r, mode, 2))) return rc;
  const long long lim = 1ll << 46;
  auto small = [lim](const int64_t* A, size_t cnt) { return std::all_of(A, A + cnt, [lim](int64_t v) { return v < lim && v > -lim; }); };
  if (!small(L, (size_t)r * m * k) || !small(R, (size_t)r * k * n) || !small(P, (size_t)r * m * n)) {
    set_error("orbit sweep (64-bit inputs): |entry| >= 2^46");
    return PLO_E_RANGE;
  }
  std::vector<long long> h;
  pack_lrp(h, m, k, n, r, L, R, P);
  const Den3 den = abs_den(denL, denR, denP);
  if (rt) {
    if (!rt_bound_ok(m, k, n, r, L, R, P)) { set_error("orbit sweep (64-bit inputs): transformed entries of %dx%dx%d may reach 2^62", m, k, n); return PLO_E_RANGE; }
    RtArgs a = rt_args(m, k, n, r, mode, measure, seed, den, false, 0);
    if (tg2) a.g2 = 1;
    return rt_sync<long long>(a, h, lo, hi, best, tnnz, tnno, tg2);
  }
  const double3 inv = inverses(den);
  with_shape(m, k, n, r, [&](auto s) {
    using S = decltype(s);
    rc = sweep_sync(h, 4, measure, lo, hi, [&](int grid, uint64_t l, uint64_t u, Key* bb, uint32_t* c0, uint32_t* c1, double* g) {
      with_mode(mode, [&](auto md) {
        orbit_wide_kernel<long long, S::M, S::K, S::N, decltype(md)::value><<<grid, kThreads>>>(r, den, inv, measure, seed, l, u, bb, c0, c1, g, no_sink());
      });
    }, best, tnnz, tnno, tg2);
  });
  return rc;
}

// Pairs of rows l, l+1 of L | R | P^T at 8-bit spacing (c_lrp2), as the four-lane kernels read them
static void pack_pairs(plo_orbit_plan* pl) {
  const int m = pl->m, k = pl->k, n = pl->n, r = pl->r, npair = (r + 1) / 2;
  pl->h_lrp2.assign((size_t)npair * (m * k + k * n + m * n), 0);
  const int* src = pl->h_lrp.data();
  int* d2 = pl->h_lrp2.data();
  const int widths[3] = {m * k, k * n, m * n};
  for (int t = 0; t < 3; ++t) {
    for (int q = 0; q < npair; ++q)
      for (int e = 0; e < widths[t]; ++e) {
        const int a0 = src[(size_t)(2 * q) * widths[t] + e];
        const int a1 = 2 * q + 1 < r ? src[(size_t)(2 * q + 1) * widths[t] + e] : 0;
        *d2++ = a0 + 256 * a1;
      }
    src += (size_t)r * widths[t];
  }
}

// Growth-factor plans of 2x2x2, r = 7 that orbit_sweep8x_kernel takes: worst-case row norm^2 up to this bound.  The kernel has no
// such limit of its own; the bound is where the routing stood when the kernel also held a sqrt table of smax + 1 entries (16
// replicas of 8 bytes each, beside 72 KB of first-stage tables, one 512-thread block in 228 KB), so that larger inputs such as
// Winograd scaled by 6 keep the four-lane kernel.
constexpr long long kTable8xMaxRowNorm2 = 1234;

// The sweep kernel of a compiled-shape plan and its launch configuration.  `narrow`: the int32 product bound holds (magnitude_ok,
// which also gave smax and the lane bounds).  Precedence: Wide, the 2x2x2 r = 7 table kernels, the four-lane kernels, Plain; a
// table or four-lane kernel that cannot run falls back as noted.
template <class S>
static int choose_path(plo_orbit_plan* pl, bool narrow, long long smax, bool lanes16, bool lanes8) {
  constexpr int M = S::M, K = S::K, N = S::N, RU = S::RU;
  constexpr size_t scratch = MaxDim2<M, K, N>::d > 2 ? (size_t)MaxDim2<M, K, N>::value * kThreads * sizeof(int) : 0;
  const int sms = sm_count();
  const bool g2 = pl->measure == PLO_MEASURE_G2, r7 = M == 2 && K == 2 && N == 2 && pl->r == 7;
  // sqrt table: covers every reachable row norm^2 when that fits in 32 KB, else the first 4096 values
  pl->lutn = narrow && g2 ? (int)std::min<long long>(smax + 1, 4096) : 0;
  pl->lutfull = narrow && g2 && smax + 1 <= 4096;
  pl->pack = narrow && lanes16;
  pl->smem = (size_t)pl->lutn * sizeof(double) + scratch;
  const SweepKernel plain0 = sweep_kernel<S, 0>(pl->measure, pl->lutfull, pl->pack), plain1 = sweep_kernel<S, 1>(pl->measure, pl->lutfull, pl->pack);
  if (pl->smem > 48 * 1024 && !(allow_smem(plain0, pl->smem) && allow_smem(plain1, pl->smem))) {
    set_error("orbit sweep: cannot reserve %zu bytes of shared memory", pl->smem);
    return PLO_E_CUDA;
  }
  pl->path = narrow ? OrbitPath::Plain : OrbitPath::Wide;
  pl->grid = sms * std::max(1, blocks_per_sm(plain1, kThreads, pl->smem));
  // four-lane kernels: every transformed entry below 128, pairs of rows packed at 8-bit spacing in c_lrp2
  const bool four = narrow && lanes8 && (long long)((pl->r + 1) / 2) * (M * K + K * N + M * N) <= kConst2Ints;
  if (g2 && four) {
    const int nb = r7 && smax <= kTable8xMaxRowNorm2 ? blocks_per_sm(&orbit_sweep8x_kernel<0>, &orbit_sweep8x_kernel<1>, kXThreads, kXTabBytes) : 0;
    if (nb > 0) {
      pl->path = OrbitPath::Table8x;
      pl->grid = sms * nb;
      pl->smem = kXTabBytes;
    } else {
      pl->path = OrbitPath::FourLaneG2;
      pl->grid = sms * std::max(1, blocks_per_sm(&orbit_sweep8_kernel<M, K, N, 0, RU>, &orbit_sweep8_kernel<M, K, N, 1, RU>, kThreads, pl->smem));
      pack_pairs(pl);
    }
  } else if (!g2 && r7 && pl->pack) {
    const int nb = blocks_per_sm(&orbit_sweep2x_kernel<0>, &orbit_sweep2x_kernel<1>, kXThreads, kX2TabBytes);
    if (nb > 0) {
      pl->path = OrbitPath::Table2x;
      pl->grid = sms * nb;
      pl->smem = kX2TabBytes;
    }
  } else if (!g2 && four && pl->den.x < 128 && pl->den.y < 128 && pl->den.z < 128) {
    const int nb = blocks_per_sm(&orbit_sweepn8_kernel<M, K, N, 0>, &orbit_sweepn8_kernel<M, K, N, 1>, kThreads, scratch);
    if (nb > 0) {
      pl->path = OrbitPath::FourLaneNnz;
      pl->grid = sms * nb;
      pl->smem = scratch;
      pack_pairs(pl);
    }
  }
  return PLO_OK;
}

namespace plo {
// A sweep of [lo,hi) sharded over the first `ndev` devices of this process (one host thread: the launches are asynchronous, so the
// devices work concurrently); `create` makes the plan on the current device (plo_orbit_plan_create, plo_orbit_plan_create_quad).
// Contiguous ascending shards, winner = lexicographic minimum with the lowest index among ties.
int orbit_sweep_sharded(int ndev, int measure, uint64_t lo, uint64_t hi, plo_orbit_best* best, const std::function<int(plo_orbit_plan**)>& create) {
  if (!best || ndev < 1 || hi < lo) { set_error("orbit sweep over devices: bad argument"); return PLO_E_ARG; }
  int have = 0, prev = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have < 1) { cudaGetLastError(); return check_device(); }
  if (ndev > have) ndev = have;
  if (ndev > kMaxDevices) ndev = kMaxDevices;
  cudaGetDevice(&prev);
  std::vector<plo_orbit_plan*> plans((size_t)ndev, nullptr);
  int rc = PLO_OK;
  const uint64_t total = hi - lo, base = total / (uint64_t)ndev, rem = total % (uint64_t)ndev;
  uint64_t a = lo;
  for (int d = 0; d < ndev && !rc; ++d) {
    const uint64_t b = a + base + ((uint64_t)d < rem ? 1 : 0);
    if (cudaSetDevice(d) != cudaSuccess) { set_error("orbit sweep over devices: cudaSetDevice(%d) failed", d); rc = PLO_E_CUDA; break; }
    rc = create(&plans[(size_t)d]);
    if (!rc) rc = plo_orbit_plan_run(plans[(size_t)d], a, b, nullptr);
    a = b;
  }
  plo_orbit_best win;
  win.index = PLO_NO_INDEX; win.nnz = 0; win.nno = 0; win.score = 0.0;
  for (int d = 0; d < ndev; ++d) {
    if (!plans[(size_t)d]) continue;
    cudaSetDevice(d);
    plo_orbit_best b;
    if (!rc) rc = plo_orbit_plan_result(plans[(size_t)d], nullptr, &b);
    if (!rc && b.index != PLO_NO_INDEX) {
      bool better = win.index == PLO_NO_INDEX;
      if (!better) {
        if (measure == PLO_MEASURE_G2) better = b.score < win.score;  // shards are ascending: ties keep the earlier shard
        else better = b.nnz < win.nnz || (b.nnz == win.nnz && b.nno < win.nno);
      }
      if (better) win = b;
    }
    plo_orbit_plan_destroy(plans[(size_t)d]);
  }
  cudaSetDevice(prev);
  if (!rc) *best = win;
  return rc;
}
}  // namespace plo

extern "C" {

uint64_t plo_orbit_space(int m, int k, int n) {
  auto one = [](int s, unsigned __int128& acc) {
    for (int i = 2; i <= s; ++i) acc *= (unsigned)i * (unsigned)i;  // two permutations
    for (int i = 0; i < s; ++i) acc *= 2u;
    for (int i = 0; i < s * (s - 1) / 2; ++i) acc *= 3u;
  };
  unsigned __int128 acc = 1;
  one(m, acc); if (acc >> 64) return 0;
  one(k, acc); if (acc >> 64) return 0;
  one(n, acc); if (acc >> 64) return 0;
  return (uint64_t)acc;
}

int plo_orbit_decode(int m, int k, int n, int mode, uint64_t seed, uint64_t index, int32_t* U, int32_t* V, int32_t* W) {
  if (!U || !V || !W || m < 1 || k < 1 || n < 1 || m > kMaxDim || k > kMaxDim || n > kMaxDim || (mode != 0 && mode != 1)) {
    set_error("plo_orbit_decode: bad argument");
    return PLO_E_ARG;
  }
  int scr[kMaxDim * kMaxDim];
  with_mode(mode, [&](auto modeTag) {
    constexpr int MODE = decltype(modeTag)::value;
    Digits<MODE> ds(seed, index);
    auto one = [&](int s, int32_t* out) {
      switch (s) {
#define CASE(S) case S: { Zoi z = decode_zoi<S, MODE>(ds); expand_zoi<S, false>(z, out, scr, 1); break; }
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
#undef CASE
      }
    };
    one(m, U); one(k, V); one(n, W);
  });
  return PLO_OK;
}

int plo_orbit_plan_create(plo_orbit_plan** plan, int m, int k, int n, int r, const int32_t* L, const int32_t* R,
                          const int32_t* P, int32_t denL, int32_t denR, int32_t denP, int measure, int mode,
                          uint64_t seed) {
  if (!plan || !L || !R || !P || r < 1 || denL == 0 || denR == 0 || denP == 0 ||
      (measure != PLO_MEASURE_NNZ && measure != PLO_MEASURE_G2) || (mode != 0 && mode != 1)) {
    set_error("plo_orbit_plan_create: bad argument");
    return PLO_E_ARG;
  }
  int rc = check_device();
  if (rc) return rc;
  bool rt = false;
  if ((rc = orbit_route(m, k, n, r, &rt)) || (rc = orbit_limits(m, k, n, r, mode, 1))) return rc;
  if (rt && !rt_bound_ok(m, k, n, r, L, R, P)) { set_error("orbit sweep: transformed entries of %dx%dx%d may reach 2^62", m, k, n); return PLO_E_RANGE; }
  long long smax = 0;
  bool lanes16 = false, lanes8 = false;
  const bool narrow = magnitude_ok(m, k, n, r, L, R, P, &smax, &lanes16, &lanes8);  // else Wide (compiled shapes)
  plo_orbit_plan* pl = new plo_orbit_plan();  // value-initialised: no device buffer, no sqrt table
  pl->m = m; pl->k = k; pl->n = n; pl->r = r; pl->measure = measure; pl->mode = mode; pl->seed = seed;
  const Den3 den = abs_den(denL, denR, denP);
  pl->den = make_int3((int)den.x, (int)den.y, (int)den.z);
  pl->inv_den = 1.0 / ((double)den.x * (double)den.y * (double)den.z);
  pl->inv_den3 = inverses(den);
  pack_lrp(pl->h_lrp, m, k, n, r, L, R, P);
  for (int i = 0; i < 10; ++i) {
    pl->h_pkeys[2 * i] = (uint32_t)seed + (uint32_t)i * 0x9E3779B9u;
    pl->h_pkeys[2 * i + 1] = (uint32_t)(seed >> 32) + (uint32_t)i * 0xBB67AE85u;
  }
  if (rt) {
    pl->path = OrbitPath::Runtime;
    pl->rta = rt_args(m, k, n, r, mode, measure, seed, den, narrow, 0);
    pl->smem = rt_smem(m, k, n);
    const int nb = rt_prepare<int>(m, k, n);
    pl->grid = sm_count() * nb;
    if (nb < 1) rc = PLO_E_CUDA;
  } else {
    with_shape(m, k, n, r, [&](auto s) { rc = choose_path<decltype(s)>(pl, narrow, smax, lanes16, lanes8); });
  }
  if (!rc && (pool_alloc(&pl->d_block_best, sizeof(Key) * pl->grid) != cudaSuccess || pool_alloc(&pl->d_out, sizeof(plo_orbit_best)) != cudaSuccess)) {
    set_error("orbit sweep: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = PLO_E_CUDA;
  }
  const bool four = pl->path == OrbitPath::FourLaneG2 || pl->path == OrbitPath::FourLaneNnz;
  if (!rc && four && m == 3 && k == 3 && n == 3) {
    // built once per plan, on the default stream (plan creation is synchronous); without it the kernels decode per candidate
    if (pool_alloc(&pl->d_z3tab, (size_t)kZ3Count * kZ3Chunks * sizeof(int4)) == cudaSuccess) {
      with_mode(mode, [&](auto md) { zoi3_table_kernel<decltype(md)::value><<<(kZ3Count + kThreads - 1) / kThreads, kThreads>>>(pl->d_z3tab); });
      if (cudaDeviceSynchronize() != cudaSuccess) { cudaGetLastError(); pool_free(pl->d_z3tab); pl->d_z3tab = nullptr; }
    } else {
      cudaGetLastError();
      pl->d_z3tab = nullptr;
    }
  }
  if (!rc && pl->path == OrbitPath::Wide && (pool_alloc(&pl->d_wide_cnt, 8) != cudaSuccess || pool_alloc(&pl->d_wide_g2, 8) != cudaSuccess)) {
    set_error("orbit sweep: device allocation failed");
    rc = PLO_E_CUDA;
  }
  if (rc) {
    plo_orbit_plan_destroy(pl);
    return rc;
  }
  *plan = pl;
  return PLO_OK;
}

int plo_orbit_plan_create_quad(plo_orbit_plan** plan, int64_t d, int m, int k, int n, int r, const int64_t* La, const int64_t* Lb,
                               const int64_t* Ra, const int64_t* Rb, const int64_t* Pa, const int64_t* Pb, int64_t denL, int64_t denR,
                               int64_t denP, int measure, int mode, uint64_t seed) {
  if (!plan || !La || !Lb || !Ra || !Rb || !Pa || !Pb || r < 1 || denL == 0 || denR == 0 || denP == 0 ||
      (measure != PLO_MEASURE_NNZ && measure != PLO_MEASURE_G2) || (mode != 0 && mode != 1)) {
    set_error("plo_orbit_plan_create_quad: bad argument");
    return PLO_E_ARG;
  }
  int rc = quad_field_ok(d, measure, "plo_orbit_plan_create_quad");
  if (rc || (rc = check_device())) return rc;
  if (m < 1 || k < 1 || n < 1 || m > kMaxDim || k > kMaxDim || n > kMaxDim) return orbit_limits(m, k, n, r, mode, 1);
  const size_t nl = (size_t)r * m * k, nr = (size_t)r * k * n, np = (size_t)r * m * n;
  const int64_t* parts[6] = {La, Lb, Ra, Rb, Pa, Pb};
  const size_t sizes[6] = {nl, nl, nr, nr, np, np};
  bool fits32 = true, small = true;  // small: the magnitude bound below is computed in int64 without overflow (at most 2^10 |entry|)
  for (int t = 0; t < 6; ++t)
    for (size_t e = 0; e < sizes[t]; ++e) {
      const int64_t v = parts[t][e];
      fits32 = fits32 && v >= INT32_MIN && v <= INT32_MAX;
      small = small && v < (1ll << 53) && v > -(1ll << 53);
    }
  if ((rc = orbit_limits(m, k, n, r, mode, fits32 ? 2 : 4))) return rc;  // both parts in the constant bank
  if (!small) { set_error("plo_orbit_plan_create_quad: |entry| >= 2^53"); return PLO_E_RANGE; }
  if (!rt_bound_ok(m, k, n, r, La, Ra, Pa) || !rt_bound_ok(m, k, n, r, Lb, Rb, Pb)) {
    set_error("plo_orbit_plan_create_quad: transformed entries of a part of %dx%dx%d may reach 2^62", m, k, n);
    return PLO_E_RANGE;
  }
  plo_orbit_plan* pl = new plo_orbit_plan();
  pl->m = m; pl->k = k; pl->n = n; pl->r = r; pl->measure = measure; pl->mode = mode; pl->seed = seed;
  pl->path = OrbitPath::Quadratic;
  pl->q64 = !fits32;
  const Den3 den = abs_den(denL, denR, denP);
  // L | R | P^T of the rational parts, then of the sqrt(d) parts
  std::vector<long long> a, b;
  pack_lrp(a, m, k, n, r, La, Ra, Pa);
  pack_lrp(b, m, k, n, r, Lb, Rb, Pb);
  a.insert(a.end(), b.begin(), b.end());
  if (fits32) {
    pl->h_lrp.assign(a.begin(), a.end());
  } else {
    pl->h_lrp.resize(a.size() * 2);
    std::memcpy(pl->h_lrp.data(), a.data(), a.size() * sizeof(long long));
  }
  pl->rta = rt_args(m, k, n, r, mode, measure, seed, den, false, 0);
  pl->sqrtd = d > 0 ? std::sqrt((double)d) : 0.0;
  pl->smem = rt_smem(m, k, n);
  const int nb = pl->q64 ? rt_prepare<long long, true>(m, k, n) : rt_prepare<int, true>(m, k, n);
  pl->grid = sm_count() * nb;
  if (nb < 1) rc = PLO_E_CUDA;
  if (!rc && (pool_alloc(&pl->d_block_best, sizeof(Key) * pl->grid) != cudaSuccess || pool_alloc(&pl->d_out, sizeof(plo_orbit_best)) != cudaSuccess)) {
    set_error("orbit sweep: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = PLO_E_CUDA;
  }
  if (rc) {
    plo_orbit_plan_destroy(pl);
    return rc;
  }
  *plan = pl;
  return PLO_OK;
}

static int orbit_upload(plo_orbit_plan* pl, cudaStream_t st) {
  bank_acquire(st, const_owner() != pl);
  if (const_owner() != pl) {
    PLO_CUDA(cudaMemcpyToSymbolAsync(c_lrp, pl->h_lrp.data(), pl->h_lrp.size() * sizeof(int), 0, cudaMemcpyHostToDevice, st));
    if (!pl->h_lrp2.empty()) PLO_CUDA(cudaMemcpyToSymbolAsync(c_lrp2, pl->h_lrp2.data(), pl->h_lrp2.size() * sizeof(int), 0, cudaMemcpyHostToDevice, st));
    PLO_CUDA(cudaMemcpyToSymbolAsync(c_pkeys, pl->h_pkeys, sizeof(pl->h_pkeys), 0, cudaMemcpyHostToDevice, st));
    if (pl->path == OrbitPath::Quadratic) PLO_CUDA(cudaMemcpyToSymbolAsync(c_sqrtd, &pl->sqrtd, sizeof(double), 0, cudaMemcpyHostToDevice, st));
    const_owner() = pl;
  }
  return PLO_OK;
}

int plo_orbit_plan_run(plo_orbit_plan* pl, uint64_t lo, uint64_t hi, void* stream) {
  if (!pl) { set_error("plo_orbit_plan_run: null plan"); return PLO_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  int rc = orbit_upload(pl, st);
  if (rc) return rc;
  // the compiled-shape kernels' winner: orbit_final_kernel reduces the block keys and re-scores it with every measure
  auto final = [&]() {
    with_plan(pl, [&](auto s, auto md) {
      using S = decltype(s);
      orbit_final_kernel<S::M, S::K, S::N, decltype(md)::value><<<1, kThreads, 0, st>>>(pl->r, pl->den, pl->seed, pl->grid, pl->measure, pl->inv_den,
                                                                                        pl->d_block_best, pl->d_out);
    });
  };
  switch (pl->path) {
    case OrbitPath::Runtime:
    case OrbitPath::Quadratic: {
      const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>(hi > lo ? (hi - lo + kThreads - 1) / kThreads : 1, (uint64_t)pl->grid));
      with_rt(pl, [&](auto ta, auto q) {
        using TA = decltype(ta);
        rt_launch<TA, decltype(q)::value>(pl->rta, grid, st, lo, hi, pl->d_block_best, nullptr, nullptr, nullptr, no_sink());
        rt_final<TA, decltype(q)::value>(pl->rta, grid, st, pl->d_block_best, pl->d_out);
      });
      break;
    }
    case OrbitPath::Wide: {
      Key none;
      none.primary = ~0ull; none.index = ~0ull;
      std::vector<Key> init((size_t)pl->grid, none);
      PLO_CUDA(cudaMemcpyAsync(pl->d_block_best, init.data(), sizeof(Key) * pl->grid, cudaMemcpyHostToDevice, st));
      if (hi > lo)
        wide_launch(pl, (int)std::min<uint64_t>((hi - lo + kThreads - 1) / kThreads, (uint64_t)pl->grid), st, lo, hi, pl->d_block_best, nullptr, nullptr,
                    nullptr, no_sink());
      break;
    }
    case OrbitPath::Table8x:
      with_mode(pl->mode, [&](auto md) {
        orbit_sweep8x_kernel<decltype(md)::value><<<pl->grid, kXThreads, pl->smem, st>>>(pl->seed, lo, hi, pl->d_block_best);
      });
      final();
      break;
    case OrbitPath::Table2x:
      with_mode(pl->mode, [&](auto md) {
        orbit_sweep2x_kernel<decltype(md)::value><<<pl->grid, kXThreads, pl->smem, st>>>(pl->den, pl->seed, lo, hi, pl->d_block_best);
      });
      final();
      break;
    case OrbitPath::FourLaneNnz:
      with_plan(pl, [&](auto s, auto md) {
        using S = decltype(s);
        orbit_sweepn8_kernel<S::M, S::K, S::N, decltype(md)::value><<<pl->grid, kThreads, pl->smem, st>>>(pl->r, pl->den, pl->seed, lo, hi, pl->d_block_best,
                                                                                                         pl->d_z3tab);
      });
      final();
      break;
    case OrbitPath::FourLaneG2:
      with_plan(pl, [&](auto s, auto md) {
        using S = decltype(s);
        orbit_sweep8_kernel<S::M, S::K, S::N, decltype(md)::value, S::RU><<<pl->grid, kThreads, pl->smem, st>>>(pl->r, pl->seed, lo, hi, pl->lutn, (int)pl->lutfull,
                                                                                                               pl->d_block_best, pl->d_z3tab);
      });
      final();
      break;
    case OrbitPath::Plain:
      with_plan(pl, [&](auto s, auto md) {
        sweep_kernel<decltype(s), decltype(md)::value>(pl->measure, pl->lutfull, pl->pack)<<<pl->grid, kThreads, pl->smem, st>>>(pl->r, pl->den, pl->seed, lo, hi,
                                                                                                                              pl->lutn, pl->d_block_best);
      });
      final();
      break;
  }
  PLO_CUDA(cudaGetLastError());
  bank_release(st);
  return PLO_OK;
}

// The winner of the last run as one slot of a world x 4 table of int64 words (order-preserving bits of the score, index, nnz,
// nno; INT64_MAX everywhere else): after an all-reduce(MIN) over the table every rank holds every local winner, and the global
// one is the lexicographic minimum -- no host round trip between the sweep and the collective.
__global__ void orbit_pack_slot_kernel(const plo_orbit_best* __restrict__ out, long long* __restrict__ slots, int rank, int world) {
  for (int w = threadIdx.x; w < world * 4; w += blockDim.x) slots[w] = 0x7fffffffffffffffll;
  __syncthreads();
  if (threadIdx.x == 0 && out->index != ~0ull && out->index <= 0x7fffffffffffffffull) {
    slots[rank * 4 + 0] = __double_as_longlong(out->score);  // score >= 0: IEEE bits order like integers
    slots[rank * 4 + 1] = (long long)out->index;
    slots[rank * 4 + 2] = out->nnz;
    slots[rank * 4 + 3] = out->nno;
  }
}

int plo_orbit_plan_pack(plo_orbit_plan* pl, int64_t* slots, int rank, int world, void* stream) {
  if (!pl || !slots || world < 1 || rank < 0 || rank >= world) { set_error("plo_orbit_plan_pack: bad argument"); return PLO_E_ARG; }
  switch (pl->path) {
    case OrbitPath::Wide:
      set_error("plo_orbit_plan_pack: the 64-bit path picks its winner on the host (use plo_orbit_plan_result)");
      return PLO_E_SHAPE;
    case OrbitPath::Runtime:
    case OrbitPath::Quadratic:
    case OrbitPath::Table8x:
    case OrbitPath::Table2x:
    case OrbitPath::FourLaneNnz:
    case OrbitPath::FourLaneG2:
    case OrbitPath::Plain:
      break;
  }
  orbit_pack_slot_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(pl->d_out, reinterpret_cast<long long*>(slots), rank, world);
  PLO_CUDA(cudaGetLastError());
  return PLO_OK;
}

int plo_set_orbit_any_shape(int enable) {
  if (enable != 0 && enable != 1) { set_error("plo_set_orbit_any_shape: need 0 or 1"); return PLO_E_ARG; }
  g_any_shape = enable;
  return PLO_OK;
}

int plo_selftest_matrix_index(void) { return matrix_index_mismatches<2, 48>() + matrix_index_mismatches<3, 7776>(); }

int plo_orbit_plan_launches(const plo_orbit_plan*) { return 2; }

int plo_orbit_magnitude_bounds(int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int64_t* bounds) {
  if (!L || !R || !P || !bounds || r < 1 || m < 1 || k < 1 || n < 1 || m > kMaxDim || k > kMaxDim || n > kMaxDim) {
    set_error("plo_orbit_magnitude_bounds: bad argument");
    return PLO_E_ARG;
  }
  long long smax = 0, b[3] = {0, 0, 0};
  bool l16 = false, l8 = false;
  const bool ok = magnitude_ok(m, k, n, r, L, R, P, &smax, &l16, &l8, b);
  bounds[0] = b[0]; bounds[1] = b[1]; bounds[2] = b[2];
  return ok ? (l8 ? 4 : (l16 ? 2 : 1)) : 0;
}

// which sweep kernel plo_orbit_plan_run launches, and how many candidate-matrix entries one 32-bit multiply-add carries in it
int plo_orbit_plan_kernel(const plo_orbit_plan* pl, char* name, int cap, int* lanes) {
  if (!pl) { set_error("plo_orbit_plan_kernel: null plan"); return PLO_E_ARG; }
  const char* nm = "";
  int ln = 1;
  // the suffix names the code variant the templates select for this shape, so that a profile is never quoted for another variant
  switch (pl->path) {
    case OrbitPath::Runtime: nm = "orbit_rt_kernel"; ln = 1; break;
    case OrbitPath::Quadratic: nm = "orbit_rt_kernel+quad"; ln = 1; break;
    case OrbitPath::Wide: nm = "orbit_wide_kernel"; ln = 1; break;
    case OrbitPath::Table8x: nm = "orbit_sweep8x_kernel"; ln = 4; break;
    case OrbitPath::Table2x: nm = "orbit_sweep2x_kernel"; ln = 2; break;
    case OrbitPath::FourLaneNnz:
      nm = pl->m * pl->k * pl->n >= 84 ? (pl->n >= 5 ? "orbit_sweepn8_kernel+3phase+tri" : "orbit_sweepn8_kernel+3phase") : "orbit_sweepn8_kernel";
      ln = 4;
      break;
    case OrbitPath::FourLaneG2: nm = pl->n >= 5 && !(pl->m == 2 && pl->k == 2 && pl->n == 2) ? "orbit_sweep8_kernel+tri" : "orbit_sweep8_kernel"; ln = 4; break;
    case OrbitPath::Plain: nm = "orbit_sweep_kernel"; ln = pl->pack ? 2 : 1; break;
  }
  if (name && cap > 0) { strncpy(name, nm, (size_t)cap - 1); name[cap - 1] = 0; }
  if (lanes) *lanes = ln;
  return PLO_OK;
}

int plo_orbit_plan_result(plo_orbit_plan* pl, void* stream, plo_orbit_best* best) {
  if (!pl || !best) { set_error("plo_orbit_plan_result: bad argument"); return PLO_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  switch (pl->path) {
    case OrbitPath::Wide: {  // host picks the winner among the block keys, one more 1-candidate launch returns all its measures
      std::vector<Key> bb((size_t)pl->grid);
      PLO_CUDA(cudaMemcpyAsync(bb.data(), pl->d_block_best, sizeof(Key) * pl->grid, cudaMemcpyDeviceToHost, st));
      PLO_CUDA(cudaStreamSynchronize(st));
      const Key b = min_key(bb);
      best->index = b.index; best->nnz = 0; best->nno = 0; best->score = 0.0;
      if (b.index == ~0ull) return PLO_OK;
      int rc = orbit_upload(pl, st);
      if (rc) return rc;
      wide_launch(pl, 1, st, b.index, b.index + 1, nullptr, pl->d_wide_cnt, pl->d_wide_cnt + 1, pl->d_wide_g2, no_sink());
      uint32_t cnt[2];
      double g2 = 0.0;
      PLO_CUDA(cudaMemcpyAsync(cnt, pl->d_wide_cnt, 8, cudaMemcpyDeviceToHost, st));
      PLO_CUDA(cudaMemcpyAsync(&g2, pl->d_wide_g2, 8, cudaMemcpyDeviceToHost, st));
      PLO_CUDA(cudaStreamSynchronize(st));
      best->nnz = cnt[0]; best->nno = cnt[1];
      best->score = pl->measure == PLO_MEASURE_G2 ? g2 : (double)cnt[0];
      return PLO_OK;
    }
    case OrbitPath::Runtime:
    case OrbitPath::Quadratic:
    case OrbitPath::Table8x:
    case OrbitPath::Table2x:
    case OrbitPath::FourLaneNnz:
    case OrbitPath::FourLaneG2:
    case OrbitPath::Plain:
      break;
  }
  PLO_CUDA(cudaMemcpyAsync(best, pl->d_out, sizeof(plo_orbit_best), cudaMemcpyDeviceToHost, st));
  PLO_CUDA(cudaStreamSynchronize(st));
  return PLO_OK;
}

void plo_orbit_plan_destroy(plo_orbit_plan* pl) {
  if (!pl) return;
  for (int d = 0; d < kMaxDevices; ++d) if (g_const_owner_dev[d] == pl) g_const_owner_dev[d] = nullptr;
  if (pl->d_block_best) pool_free(pl->d_block_best);
  if (pl->d_out) pool_free(pl->d_out);
  pool_free(pl->d_wide_cnt); pool_free(pl->d_wide_g2); pool_free(pl->d_z3tab);
  delete pl;
}

int plo_orbit_sweep(uint32_t p, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P,
                    int32_t denL, int32_t denR, int32_t denP, int measure, int mode, uint64_t seed, uint64_t lo,
                    uint64_t hi, plo_orbit_best* best) {
  if (!best) { set_error("plo_orbit_sweep: null output"); return PLO_E_ARG; }
  if (p != 0) {
    if (measure != PLO_MEASURE_NNZ) { set_error("plo_orbit_sweep: only the sparsity measure exists over Z/pZ (src/orbiter.cpp:426)"); return PLO_E_ARG; }
    return orbit_modp(p, m, k, n, r, L, R, P, mode, seed, lo, hi, best, nullptr, nullptr);
  }
  plo_orbit_plan* pl = nullptr;
  int rc = plo_orbit_plan_create(&pl, m, k, n, r, L, R, P, denL, denR, denP, measure, mode, seed);
  if (rc) return rc;
  rc = plo_orbit_plan_run(pl, lo, hi, nullptr);
  if (!rc) rc = plo_orbit_plan_result(pl, nullptr, best);
  plo_orbit_plan_destroy(pl);
  return rc;
}

// The same sweep sharded over the first `ndev` devices of this process (orbit_sweep_sharded).
int plo_orbit_sweep_devices(int ndev, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int32_t denL,
                            int32_t denR, int32_t denP, int measure, int mode, uint64_t seed, uint64_t lo, uint64_t hi,
                            plo_orbit_best* best) {
  if (!best || ndev < 1 || hi < lo) { set_error("plo_orbit_sweep_devices: bad argument"); return PLO_E_ARG; }
  return orbit_sweep_sharded(ndev, measure, lo, hi, best, [&](plo_orbit_plan** pl) {
    return plo_orbit_plan_create(pl, m, k, n, r, L, R, P, denL, denR, denP, measure, mode, seed);
  });
}

// Both measures of every candidate of [lo,hi) on the default stream: per-candidate tables and/or the survivor sink armed.
static void table_launch(const plo_orbit_plan* pl, int grid, uint64_t lo, uint64_t hi, uint32_t* nnz, uint32_t* nno, double* g2, Sink sink) {
  switch (pl->path) {
    case OrbitPath::Runtime:
    case OrbitPath::Quadratic: {
      RtArgs a = pl->rta;
      a.g2 = pl->path == OrbitPath::Runtime || pl->sqrtd > 0.0;  // G2 over Q(sqrt d) needs the real embedding: d > 0
      with_rt(pl, [&](auto ta, auto q) { rt_launch<decltype(ta), decltype(q)::value>(a, grid, nullptr, lo, hi, pl->d_block_best, nnz, nno, g2, sink); });
      break;
    }
    case OrbitPath::Wide:
      wide_launch(pl, grid, nullptr, lo, hi, nullptr, nnz, nno, g2, sink);
      break;
    case OrbitPath::Table8x:
    case OrbitPath::Table2x:
    case OrbitPath::FourLaneNnz:
    case OrbitPath::FourLaneG2:
    case OrbitPath::Plain:
      with_plan(pl, [&](auto s, auto md) {
        using S = decltype(s);
        orbit_table_kernel<S::M, S::K, S::N, decltype(md)::value><<<grid, kThreads>>>(pl->r, pl->den, pl->seed, lo, hi, pl->inv_den, nnz, nno, g2, sink);
      });
      break;
  }
}

// The per-candidate tables of [lo,hi) through a plan's table kernel; destroys the plan.
static int plan_table(plo_orbit_plan* pl, uint64_t lo, uint64_t hi, uint32_t* nnz, uint32_t* nno, double* g2) {
  int rc = PLO_OK;
  const size_t cnt = (size_t)(hi - lo);
  uint32_t *d_nnz = nullptr, *d_nno = nullptr;
  double* d_g2 = nullptr;
  auto cleanup = [&]() { pool_free(d_nnz); pool_free(d_nno); pool_free(d_g2); plo_orbit_plan_destroy(pl); };
  if (cnt) {
    if (pool_alloc(&d_nnz, cnt * 4) != cudaSuccess || pool_alloc(&d_nno, cnt * 4) != cudaSuccess || pool_alloc(&d_g2, cnt * 8) != cudaSuccess) {
      set_error("plo_orbit_table: cudaMalloc failed"); cleanup(); return PLO_E_CUDA;
    }
    rc = orbit_upload(pl, nullptr);
    if (!rc) {
      size_t blocks = (cnt + kThreads - 1) / kThreads;
      table_launch(pl, (int)(blocks < (size_t)pl->grid ? blocks : (size_t)pl->grid), lo, hi, d_nnz, d_nno, d_g2, no_sink());
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { set_error("plo_orbit_table: %s", cudaGetErrorString(e)); rc = PLO_E_CUDA; }
    }
    if (!rc) {
      if (nnz) cudaMemcpy(nnz, d_nnz, cnt * 4, cudaMemcpyDeviceToHost);
      if (nno) cudaMemcpy(nno, d_nno, cnt * 4, cudaMemcpyDeviceToHost);
      if (g2) cudaMemcpy(g2, d_g2, cnt * 8, cudaMemcpyDeviceToHost);
    }
  }
  cleanup();
  return rc;
}

int plo_orbit_table(int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int32_t denL,
                    int32_t denR, int32_t denP, int mode, uint64_t seed, uint64_t lo, uint64_t hi, uint32_t* nnz,
                    uint32_t* nno, double* g2) {
  if (hi < lo) { set_error("plo_orbit_table: hi < lo"); return PLO_E_ARG; }
  plo_orbit_plan* pl = nullptr;
  const int rc = plo_orbit_plan_create(&pl, m, k, n, r, L, R, P, denL, denR, denP, PLO_MEASURE_G2, mode, seed);
  return rc ? rc : plan_table(pl, lo, hi, nnz, nno, g2);
}

int plo_orbit_table_quad(int64_t d, int m, int k, int n, int r, const int64_t* La, const int64_t* Lb, const int64_t* Ra, const int64_t* Rb,
                         const int64_t* Pa, const int64_t* Pb, int64_t denL, int64_t denR, int64_t denP, int mode, uint64_t seed, uint64_t lo,
                         uint64_t hi, uint32_t* nnz, uint32_t* nno, double* g2) {
  if (hi < lo) { set_error("plo_orbit_table_quad: hi < lo"); return PLO_E_ARG; }
  if (g2 && d < 0) { set_error("plo_orbit_table_quad: G2 needs a real embedding of Q(sqrt %lld), d > 0 (pass g2 = NULL)", (long long)d); return PLO_E_ARG; }
  plo_orbit_plan* pl = nullptr;
  const int rc = plo_orbit_plan_create_quad(&pl, d, m, k, n, r, La, Lb, Ra, Rb, Pa, Pb, denL, denR, denP, d > 0 ? PLO_MEASURE_G2 : PLO_MEASURE_NNZ,
                                            mode, seed);
  return rc ? rc : plan_table(pl, lo, hi, nnz, nno, g2);
}

// Survivors of [lo,hi): every candidate whose score does not exceed `threshold` (sparsity plans: (nnz, nno) <= (threshold.nnz,
// threshold.nno) lexicographically; growth-factor plans: score <= threshold.score), with both measures, sorted by index.
// Synchronous.  *count = number found; more than `capacity` -> PLO_E_RANGE (nothing is written; retry with *count records).
// Survivors through the plan's own (packed, table-driven, ...) sweep kernel: pass 1 = the sweep with the constant-bank sink armed
// (indices only, 8 bytes per survivor), device radix sort of the indices, pass 2 = both measures of the survivors in index order.
// The growth-factor threshold is applied to the kernel's unscaled key with two ulps of slack and exactly on the records afterwards.
static int survivors_from_the_sweep(plo_orbit_plan* pl, uint64_t lo, uint64_t hi, const plo_orbit_best* threshold, uint64_t capacity,
                                    plo_orbit_best* out, uint64_t* count) {
  const uint64_t cap = capacity ? capacity : 1;
  unsigned long long *d_idx = nullptr, *d_sorted = nullptr, *d_cnt = nullptr;
  uint4* d_rec = nullptr;
  void* d_temp = nullptr;
  size_t temp_bytes = 0;
  auto cleanup = [&]() { pool_free(d_idx); pool_free(d_sorted); pool_free(d_cnt); pool_free(d_rec); pool_free(d_temp); };
  cub::DeviceRadixSort::SortKeys(nullptr, temp_bytes, d_idx, d_sorted, (int)std::min<uint64_t>(cap, 0x7fffffffull));
  if (cap > 0x7fffffffull || pool_alloc(&d_idx, cap * 8) != cudaSuccess || pool_alloc(&d_sorted, cap * 8) != cudaSuccess || pool_alloc(&d_cnt, 8) != cudaSuccess ||
      pool_alloc(&d_rec, cap * 32) != cudaSuccess || pool_alloc(&d_temp, temp_bytes ? temp_bytes : 1) != cudaSuccess) {
    set_error("plo_orbit_plan_survivors: device allocation for %llu records failed", (unsigned long long)cap);
    cleanup();
    return PLO_E_CUDA;
  }
  Surv sv;
  if (pl->measure == PLO_MEASURE_G2) {
    double raw = threshold->score / pl->inv_den;
    raw = std::nextafter(std::nextafter(raw, INFINITY), INFINITY);
    if (!(raw >= 0.0)) raw = 0.0;
    std::memcpy(&sv.thr, &raw, 8);
  } else {
    sv.thr = ((unsigned long long)threshold->nnz << 32) | threshold->nno;
  }
  sv.idx = d_idx; sv.count = d_cnt; sv.cap = capacity;
  const Surv off{0ull, nullptr, nullptr, 0ull};
  bank_acquire(nullptr, true);  // nothing that still reads the bank may see the sink armed
  cudaError_t e = cudaMemset(d_cnt, 0, 8);
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_surv, &sv, sizeof(sv));
  int rc = PLO_OK;
  if (e == cudaSuccess) rc = plo_orbit_plan_run(pl, lo, hi, nullptr);
  cudaError_t e2 = cudaMemcpyToSymbol(c_surv, &off, sizeof(off));  // always disarm (synchronises with the sweep)
  if (e == cudaSuccess) e = e2;
  unsigned long long found = 0;
  if (e == cudaSuccess && rc == PLO_OK) e = cudaMemcpy(&found, d_cnt, 8, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess || rc != PLO_OK) {
    if (e != cudaSuccess) { set_error("plo_orbit_plan_survivors: %s", cudaGetErrorString(e)); rc = PLO_E_CUDA; }
    cleanup();
    return rc;
  }
  *count = found;
  if (found > capacity) {
    set_error("plo_orbit_plan_survivors: %llu survivors, capacity %llu", found, (unsigned long long)capacity);
    cleanup();
    return PLO_E_RANGE;
  }
  std::vector<uint4> rec((size_t)found * 2);
  if (found) {
    e = cub::DeviceRadixSort::SortKeys(d_temp, temp_bytes, d_idx, d_sorted, (int)found);
    if (e == cudaSuccess) {
      const int grid = (int)std::min<uint64_t>((found + kThreads - 1) / kThreads, (uint64_t)sm_count() * 8);
      with_plan(pl, [&](auto s, auto md) {
        using S = decltype(s);
        orbit_gather_kernel<S::M, S::K, S::N, decltype(md)::value><<<grid, kThreads>>>(pl->r, pl->den, pl->seed, d_sorted, found, pl->inv_den, d_rec);
      });
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(rec.data(), d_rec, (size_t)found * 32, cudaMemcpyDeviceToHost);
  }
  cleanup();
  if (e != cudaSuccess) { set_error("plo_orbit_plan_survivors: %s", cudaGetErrorString(e)); return PLO_E_CUDA; }
  uint64_t kept = 0;
  for (size_t i = 0; i < (size_t)found; ++i) {
    const uint4 a = rec[2 * i], b = rec[2 * i + 1];
    const unsigned long long sb = ((unsigned long long)b.y << 32) | b.x;
    double sc;
    std::memcpy(&sc, &sb, 8);
    if (pl->measure == PLO_MEASURE_G2 && !(sc <= threshold->score)) continue;  // the two ulps of slack of pass 1
    out[kept].index = ((uint64_t)a.y << 32) | a.x;
    out[kept].nnz = a.z; out[kept].nno = a.w; out[kept].score = sc;
    ++kept;
  }
  *count = kept;
  return PLO_OK;
}

int plo_orbit_plan_survivors(plo_orbit_plan* pl, uint64_t lo, uint64_t hi, const plo_orbit_best* threshold, uint64_t capacity,
                             plo_orbit_best* out, uint64_t* count) {
  if (!pl || !threshold || !count || hi < lo || (capacity && !out)) { set_error("plo_orbit_plan_survivors: bad argument"); return PLO_E_ARG; }
  *count = 0;
  if (hi == lo) return PLO_OK;
  int rc = orbit_upload(pl, nullptr);
  if (rc) return rc;
  // the compiled-shape sweep kernels emit survivors into the constant-bank sink; the 64-bit and runtime-shape kernels take a sink argument
  switch (pl->path) {
    case OrbitPath::Runtime:
    case OrbitPath::Quadratic:
    case OrbitPath::Wide:
      break;
    case OrbitPath::Table8x:
    case OrbitPath::Table2x:
    case OrbitPath::FourLaneNnz:
    case OrbitPath::FourLaneG2:
    case OrbitPath::Plain:
      return survivors_from_the_sweep(pl, lo, hi, threshold, capacity, out, count);
  }
  const uint64_t cap = capacity ? capacity : 1;
  uint4* d_rec = nullptr;
  unsigned long long* d_cnt = nullptr;
  auto cleanup = [&]() { pool_free(d_rec); pool_free(d_cnt); };
  if (pool_alloc(&d_rec, cap * 32) != cudaSuccess || pool_alloc(&d_cnt, 8) != cudaSuccess) {
    set_error("plo_orbit_plan_survivors: device allocation of %llu records failed", (unsigned long long)cap);
    cleanup();
    return PLO_E_CUDA;
  }
  cudaError_t e = cudaMemset(d_cnt, 0, 8);
  Sink sk;
  sk.rec = d_rec; sk.count = d_cnt; sk.cap = capacity;
  sk.thr_key = ((unsigned long long)threshold->nnz << 32) | threshold->nno;
  sk.thr_score = threshold->score;
  sk.measure = pl->measure;
  const uint64_t blocks = (hi - lo + kThreads - 1) / kThreads;
  const int grid = (int)std::min<uint64_t>(blocks, (uint64_t)pl->grid);
  if (e == cudaSuccess) {
    table_launch(pl, (int)std::min<uint64_t>(blocks, (uint64_t)pl->grid), lo, hi, nullptr, nullptr, nullptr, sk);
    e = cudaGetLastError();
  }
  unsigned long long found = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&found, d_cnt, 8, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) { set_error("plo_orbit_plan_survivors: %s", cudaGetErrorString(e)); cleanup(); return PLO_E_CUDA; }
  *count = found;
  if (found > capacity) {
    set_error("plo_orbit_plan_survivors: %llu survivors, capacity %llu", found, (unsigned long long)capacity);
    cleanup();
    return PLO_E_RANGE;
  }
  std::vector<uint4> rec((size_t)found * 2);
  if (found) e = cudaMemcpy(rec.data(), d_rec, (size_t)found * 32, cudaMemcpyDeviceToHost);
  cleanup();
  if (e != cudaSuccess) { set_error("plo_orbit_plan_survivors: %s", cudaGetErrorString(e)); return PLO_E_CUDA; }
  for (size_t i = 0; i < (size_t)found; ++i) {
    const uint4 a = rec[2 * i], b = rec[2 * i + 1];
    out[i].index = ((uint64_t)a.y << 32) | a.x;
    out[i].nnz = a.z; out[i].nno = a.w;
    const unsigned long long sb = ((unsigned long long)b.y << 32) | b.x;
    double sc;
    std::memcpy(&sc, &sb, 8);
    out[i].score = sc;
  }
  std::sort(out, out + found, [](const plo_orbit_best& x, const plo_orbit_best& y) { return x.index < y.index; });
  return PLO_OK;
}

int plo_orbit_sweep64(int m, int k, int n, int r, const int64_t* L, const int64_t* R, const int64_t* P, int64_t denL, int64_t denR, int64_t denP,
                      int measure, int mode, uint64_t seed, uint64_t lo, uint64_t hi, plo_orbit_best* best) {
  if (!best) { set_error("plo_orbit_sweep64: null output"); return PLO_E_ARG; }
  return orbit_wide64(m, k, n, r, L, R, P, denL, denR, denP, measure, mode, seed, lo, hi, best, nullptr, nullptr, nullptr);
}

int plo_orbit_table64(int m, int k, int n, int r, const int64_t* L, const int64_t* R, const int64_t* P, int64_t denL, int64_t denR, int64_t denP,
                      int mode, uint64_t seed, uint64_t lo, uint64_t hi, uint32_t* nnz, uint32_t* nno, double* g2) {
  return orbit_wide64(m, k, n, r, L, R, P, denL, denR, denP, PLO_MEASURE_G2, mode, seed, lo, hi, nullptr, nnz ? nnz : nullptr, nno, g2);
}

int plo_orbit_table_modp(uint32_t p, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int mode,
                         uint64_t seed, uint64_t lo, uint64_t hi, uint32_t* nnz, uint32_t* nno) {
  return orbit_modp(p, m, k, n, r, L, R, P, mode, seed, lo, hi, nullptr, nnz, nno);
}

}  // extern "C"
