// factor_sweep.cu -- random-restart search of  PLinOpt::Factorizer / backSolver
// (include/plinopt_sparsify.inl:755-867, 924-990) on sm_100a.
//
// One candidate = one random row order S of M (r x n, full column rank).
// backSolver, restated (:773-866):
//   * walk the rows in the order S, keep the first n independent ones; a kept row
//     found at position j is swapped to position i  (T.permute(i,j); swap(M[i],M[j]) :786-797);
//   * CoB = rows at positions 0..k-1 (the n independent ones + k-n "extra" rows, :803-805);
//   * every other row is solved for:  x . CoB = row  (:842-850).  With B = the n independent
//     rows, x = [row . B^-1 | 0]  (the coordinates on the extra rows are the free variables of
//     the solve and are set to zero -- the documented rule that stands in for LinBox's
//     GaussDomain::solve, DESIGN.md section 2);
//   * score = (nnz(Res), #entries of Res not in {0,+-1}, nnz(CoB))  (:863-864), minimised
//     lexicographically (tricOpCount :914-921), lowest candidate index among ties.
//
// Mapping: one group of W lanes per candidate, lane j = column j (n <= W <= 32).  The independent
// rows are kept as a reduced row echelon basis R together with the transformation T (R = T.B),
// both column-distributed in registers (lane j holds R[.][j] and T[.][j]) and both multiplied by
// ONE common non-zero scale S instead of being normalised: the kernel never divides.  A row v is
// reduced with n broadcast loads (c_i = v[pivot column i], all independent because the basis is
// *reduced*) + n lazy multiply-adds per lane (exact 96-bit accumulation, one reduction):
// S.vr = S.v - sum c_i (S R_i).  Accepting it with pivot S.pv multiplies the scale by S.pv:
// S R_i <- (S pv)(S R_i) - (S R_i)[pivot column] (S vr), new row S (S vr)  -- two products under one
// Montgomery reduction per entry, all independent (round 1 normalised the pivot instead: a Fermat
// inversion, a serial chain of 38 multiplications, per accepted row; ncu: `wait` 3.5, issue 0.54).
// The score needs no division either: a coordinate x of a solved row is 0, 1 or -1 iff S.x is 0,
// S or -S.  Arithmetic: Montgomery residues mod an odd p < 2^31.
// Rationals are scored modulo p on the device; the host layer recomputes the winner over Q
// (plo_factorizer, host_api.cpp) and verifies the score.
#include <algorithm>
#include <vector>

#include "plo_device.cuh"

namespace plo {

constexpr int kFsWarps = 4;  // candidates in flight per block
constexpr int kFsThreads = kFsWarps * 32;
constexpr int kFsMaxRows = 256;

struct FsParams {
  uint32_t p, pinv, one, one2;  // pinv = -p^-1 mod 2^32; one = R mod p (Montgomery form of 1), one2 = R^2 mod p (the form M is stored in)
  unsigned long long M64;       // floor((2^64-1)/p)
  int r, n, k;
  unsigned long long seed;
};

__device__ __forceinline__ uint32_t mont_mul(uint32_t a, uint32_t b, uint32_t p, uint32_t pinv) {
  const unsigned long long x = (unsigned long long)a * b;
  const uint32_t m = (uint32_t)x * pinv;
  const uint32_t t = (uint32_t)((x + (unsigned long long)m * p) >> 32);  // < 2p, no overflow for p < 2^31
  return t >= p ? t - p : t;
}
__device__ __forceinline__ uint32_t sub_mod(uint32_t a, uint32_t b, uint32_t p) { return a >= b ? a - b : a + p - b; }

struct FsAcc {
  unsigned long long lo;  // bits 0..63: one aligned register pair, so that the multiply-add below is a single IMAD.WIDE with carry-out
  unsigned int hi;        // bits 64..95
};
__device__ __forceinline__ void fs_mac(FsAcc& a, unsigned int x, unsigned int y) {
  asm volatile(
      "{\n\t"
      ".reg .u32 l, h;\n\t"
      "mov.b64 {l, h}, %0;\n\t"
      "mad.lo.cc.u32 l, %2, %3, l;\n\t"
      "madc.hi.cc.u32 h, %2, %3, h;\n\t"
      "addc.u32 %1, %1, 0;\n\t"
      "mov.b64 %0, {l, h};\n\t"
      "}"
      : "+l"(a.lo), "+r"(a.hi)
      : "r"(x), "r"(y));
}
__device__ __forceinline__ uint32_t fs_lds(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// The matrix M sits in shared memory times R^2 (R = 2^32), the basis in registers times R: a lazily accumulated sum of products
// sum m_i x_i carries R^3, and two REDC steps of 32 bits bring it to (sum m_i x_i) R -- the Montgomery form the basis is kept in --
// in 10 instructions (round 1: two Barrett reductions and one REDC, 51).  A < 33 p^2 < 2^67.
__device__ __forceinline__ uint32_t fs_reduce(const FsAcc& a, const FsParams& P) {
  const unsigned long long lo = a.lo;
  const uint32_t m1 = (uint32_t)a.lo * P.pinv;
  const unsigned long long mp1 = (unsigned long long)m1 * P.p;
  const unsigned long long s1 = lo + mp1;                                                                  // low 32 bits vanish
  const unsigned long long t = (s1 >> 32) + ((unsigned long long)(a.hi + (s1 < mp1 ? 1u : 0u)) << 32);     // (A + m1 p) / 2^32 < 2^36
  const uint32_t m2 = (uint32_t)t * P.pinv;
  const unsigned long long u = (t + (unsigned long long)m2 * P.p) >> 32;                                   // < 2^36 + 2^63: no overflow; u < p (1 + 2^-26)
  return (uint32_t)(u >= P.p ? u - P.p : u);
}
// (a b + c d) R^-1 mod p for Montgomery residues a, b, c, d <= p: both products under one reduction (a b + c d < 2^63, m p < 2^63)
__device__ __forceinline__ uint32_t mont_mul2(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t p, uint32_t pinv) {
  const unsigned long long x = (unsigned long long)a * b + (unsigned long long)c * d;
  const uint32_t m = (uint32_t)x * pinv;
  const uint32_t t = (uint32_t)((x + (unsigned long long)m * p) >> 32);  // < 2p
  return t >= p ? t - p : t;
}

// Philox digit stream of the row order (same definition as the orbit decode, DESIGN.md section 3)
struct FsDigits {
  unsigned long long index, seed;
  uint32_t x, R, nwords;
  uint32_t buf[4];
  __host__ __device__ __forceinline__ FsDigits(unsigned long long seed_, unsigned long long index_) : index(index_), seed(seed_), x(0), R(0), nwords(0) {}
  __host__ __device__ __forceinline__ void new_word() {
    if ((nwords & 3u) == 0) philox4x32_10((uint32_t)index, (uint32_t)(index >> 32), nwords >> 2, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), buf);
    x = buf[nwords & 3u];
    ++nwords;
    R = 1;
  }
  __host__ __device__ __forceinline__ uint32_t digit(uint32_t radix) {
    if (R == 0 || R * radix > (1u << 20)) new_word();
    const unsigned long long t = (unsigned long long)x * radix;
    x = (uint32_t)t;
    R *= radix;
    return (uint32_t)(t >> 32);
  }
};

// score key: nnz(Res) << 40 | nno(Res) << 20 | nnz(CoB)
__host__ __device__ __forceinline__ unsigned long long fs_pack(uint32_t nnz_alt, uint32_t nno_alt, uint32_t nnz_cob) {
  return ((unsigned long long)nnz_alt << 40) | ((unsigned long long)nno_alt << 20) | nnz_cob;
}

constexpr int kFsStride = 33;  // row stride of M in shared memory (words): candidates of one warp read different rows

// W lanes per candidate (W = 4, 8, 16 or 32 >= N): a warp carries 32 / W candidates side by side, each group of W lanes doing
// exactly what the comments below say for "the warp" of the W = 32 case; ballots are cut into per-group masks, shuffles use
// width W, and the data-dependent steps (row dependent / accepted, unit pivot / inversion) are predicated per group.
template <int N, int W>
#ifndef PLO_FS_MINB
#define PLO_FS_MINB 1
#endif
__global__ void __launch_bounds__(kFsThreads, PLO_FS_MINB) factor_sweep_kernel(const FsParams P, const uint32_t* __restrict__ Mg /* r x 32, times R^2 */,
                                                                  const uint32_t* __restrict__ rownnz_g, unsigned long long lo,
                                                                  unsigned long long hi, Key* __restrict__ block_best,
                                                                  uint32_t* __restrict__ table /* 3 x (hi-lo) or null */) {
  constexpr int G = 32 / W;
  constexpr unsigned kFull = 0xffffffffu;
  constexpr unsigned kGroupMask = W == 32 ? 0xffffffffu : ((1u << (W & 31)) - 1u);
  extern __shared__ uint32_t fs_smem[];
  uint32_t* Msh = fs_smem;                                  // r x kFsStride
  uint32_t* nnzsh = Msh + (size_t)P.r * kFsStride;          // r
  unsigned char* permall = reinterpret_cast<unsigned char*>(nnzsh + P.r);
  __shared__ Key red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / W, j = lane % W;                   // group within the warp, column within the group
  const int gshift = sub * W;
  unsigned char* perm = permall + (size_t)(warp * G + sub) * kFsMaxRows;
  for (int e = threadIdx.x; e < P.r * 32; e += kFsThreads) Msh[(e >> 5) * kFsStride + (e & 31)] = Mg[e];
  for (int e = threadIdx.x; e < P.r; e += kFsThreads) nnzsh[e] = rownnz_g[e];
  __syncthreads();
  uint32_t msh_a;  // 32-bit shared address of M, opaque: ptxas otherwise re-derives the generic pointer (S2R + LEA) inside the row loops
  asm volatile("mov.u32 %0, %1;" : "=r"(msh_a) : "r"((uint32_t)__cvta_generic_to_shared(Msh)));

  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  const unsigned long long step = (unsigned long long)gridDim.x * kFsWarps * G;
  for (unsigned long long base = lo + ((unsigned long long)blockIdx.x * kFsWarps + warp) * G; base < hi; base += step) {
    const unsigned long long idx = base + (unsigned)sub;
    const bool valid = idx < hi;
    // ---- row order S: Fisher-Yates from the digit stream (every lane of the group computes the digits, its first lane swaps) ----
    for (int t = j; t < P.r; t += W) perm[t] = (unsigned char)t;
    __syncwarp();
    {
      FsDigits ds(P.seed, idx);
      for (int i = 0; i + 1 < P.r; ++i) {
        const uint32_t d = ds.digit((uint32_t)(P.r - i));
        if (j == 0 && d) { const unsigned char a = perm[i]; perm[i] = perm[i + d]; perm[i + d] = a; }
      }
    }
    __syncwarp();
    // ---- selection pass: reduced echelon basis with transformation, column-distributed, kept NEGATED and times the scale S:
    //      Rj[i] = -S R_i[j], Tj[i] = -S T_i[j]  (additions only in the reduction below) ----
    uint32_t Rj[N], Tj[N];
    uint32_t pc[N];  // byte offset of the pivot column inside a row of Msh
#pragma unroll
    for (int i = 0; i < N; ++i) { Rj[i] = 0; Tj[i] = 0; pc[i] = 0; }
    int nb = 0;
    uint32_t S = P.one;
    for (int t = 0; t < P.r; ++t) {
      const bool active = valid && nb < P.n;
      if (!__any_sync(kFull, active)) break;
      const int row = perm[t];
      const uint32_t rowa = msh_a + (uint32_t)row * (kFsStride * 4);  // shared address of the row
      const uint32_t v = fs_lds(rowa + 4u * (uint32_t)j);
      FsAcc ar, at;
      ar.lo = 0; ar.hi = 0;
      at.lo = 0; at.hi = 0;
      fs_mac(ar, S, v);                         // S v
      fs_mac(at, S, j == nb ? P.one2 : 0u);     // S e_nb (times R^2, like the entries of M)
#pragma unroll
      for (int i = 0; i < N; ++i)
        if (i < nb) {
          const uint32_t c = fs_lds(rowa + pc[i]);  // v[pivot column i]: one address per group (broadcast LDS)
          fs_mac(ar, c, Rj[i]);
          fs_mac(at, c, Tj[i]);
        }
      const uint32_t vr = fs_reduce(ar, P);  // S (v - sum c_i R_i)
      const unsigned nzmask = (__ballot_sync(kFull, active && vr != 0) >> gshift) & kGroupMask;
      const bool accept = nzmask != 0;  // else: dependent on the rows kept so far (or nothing left to do for this group)
      if (!__any_sync(kFull, accept)) continue;
      const uint32_t vt = fs_reduce(at, P);  // S (e_nb - sum c_i T_i)
      // pivot: the first non-zero coordinate.  The coordinates x of the solved rows do not depend on this choice (x.B = row has one solution).
      const int pcn = accept ? __ffs(nzmask) - 1 : 0;
      const uint32_t pv = __shfl_sync(kFull, vr, pcn, W);  // S pv: the scale becomes S (S pv)
      const uint32_t nvr = vr ? P.p - vr : 0u, nvt = vt ? P.p - vt : 0u;
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const uint32_t f = __shfl_sync(kFull, Rj[i], pcn, W);  // -S R_i[pivot column]
        if (accept && i < nb) {
          // -S' R_i = (S pv)(-S R_i) - (-S R_i[pcn])(-S vr) = pv Rj[i] + f nvr
          Rj[i] = mont_mul2(pv, Rj[i], f, nvr, P.p, P.pinv);
          Tj[i] = mont_mul2(pv, Tj[i], f, nvt, P.p, P.pinv);
        }
        if (accept && i == nb) { Rj[i] = mont_mul(S, nvr, P.p, P.pinv); Tj[i] = mont_mul(S, nvt, P.p, P.pinv); pc[i] = 4u * (uint32_t)pcn; }  // -S' w = -S (S vr)
      }
      if (accept) S = mont_mul(S, pv, P.p, P.pinv);
      if (accept && j == 0 && t != nb) { const unsigned char a = perm[nb]; perm[nb] = perm[t]; perm[t] = a; }  // :793-796
      nb += accept ? 1 : 0;
    }
    __syncwarp();
    // ---- score ----
    const bool ok = valid && nb == P.n;
    uint32_t nnz_alt = 0, nno_alt = 0, nnz_cob = 0;
    if (__any_sync(kFull, ok)) {
      for (int t = 0; t < P.r; ++t) {
        const int row = perm[t];
        if (t < P.k) { nnz_alt += 1; nnz_cob += nnzsh[row]; continue; }  // identity row of Res, row of CoB
        FsAcc ax;
        ax.lo = 0; ax.hi = 0;
        const uint32_t rowa = msh_a + (uint32_t)row * (kFsStride * 4);
#pragma unroll
        for (int i = 0; i < N; ++i) fs_mac(ax, fs_lds(rowa + pc[i]), Tj[i]);  // rows i >= n of T are zero: no guard needed
        const uint32_t x = fs_reduce(ax, P);  // -S times the coordinate of `row` on the j-th independent row
        const bool nz = j < P.n && x != 0;
        nnz_alt += __popc((__ballot_sync(kFull, nz) >> gshift) & kGroupMask);
        nno_alt += __popc((__ballot_sync(kFull, nz && x != S && x != P.p - S) >> gshift) & kGroupMask);  // not +-1: neither -S nor S
      }
    }
    const unsigned long long key = ok ? fs_pack(nnz_alt, nno_alt, nnz_cob) : ~0ull;
    if (table && j == 0 && valid) {
      const unsigned long long o = (idx - lo) * 3;
      table[o] = ok ? nnz_alt : 0xffffffffu; table[o + 1] = nno_alt; table[o + 2] = nnz_cob;
    }
    if (valid && (key < best.primary || (key == best.primary && idx < best.index))) { best.primary = key; best.index = idx; }
    __syncwarp();
  }
  // lanes of a group hold the same `best`: minimum over the groups of the warp, then over the warps of the block
#pragma unroll
  for (int d = W; d < 32; d <<= 1) {
    Key o;
    o.primary = __shfl_xor_sync(kFull, best.primary, d);
    o.index = __shfl_xor_sync(kFull, best.index, d);
    if (key_less(o, best)) best = o;
  }
  if (lane == 0) red[warp] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    Key b = red[0];
    for (int w = 1; w < kFsWarps; ++w) if (key_less(red[w], b)) b = red[w];
    block_best[blockIdx.x] = b;
  }
}

// ---- factor_wide_kernel: the same candidate for 1 <= n <= 64 columns and up to 512 rows ----
// factor_sweep_kernel keeps R[.][j], T[.][j] and the pivot offsets in registers (3N words per lane) and the row order in bytes; at
// 64 columns that is beyond the register file.  Here one warp scores one candidate, lane j owns the C columns j + 32 c (C = 1 for
// n <= 32, 2 above), and the basis R, its transformation T and the pivot offsets sit in the warp's slice of shared memory:
// R[i][j][c] at word (i 32 + j) C + c, so lane j reads its C words of a row with one vector load and the 32 lanes touch 32 C
// consecutive words (no bank conflict).  The one value a lane needs from another column, R[i][pivot column] in the rank-1
// update, comes by shuffle from the lane that loaded it: no lane ever reads a word that another lane writes.  The row order is
// uint16_t.  M (r x 32 C, at most 128 KB) is read through the read-only cache, not copied to shared memory: the shared memory it
// would take holds more warps, and that measured faster on every tested shape (DESIGN.md section 5.5).  Arithmetic, digit
// stream, selection, solve rule and score are factor_sweep_kernel's.
constexpr int kFwMaxCols = 64;
constexpr int kFwMaxRows = 512;
constexpr int kFwMaxWarps = 16;  // candidates in flight per block

// words of one warp's slice: R and T (n x 32 x C each), n pivot offsets, r uint16_t of row order; a multiple of 4 (16-byte aligned)
__host__ __device__ __forceinline__ size_t fw_warp_words(int r, int n, int C) {
  return ((size_t)2 * n * 32 * C + n + (size_t)(r + 1) / 2 + 3) & ~(size_t)3;
}
__host__ __device__ __forceinline__ size_t fw_fixed_words(int r) { return ((size_t)r + 3) & ~(size_t)3; }  // the row nnz

__device__ __forceinline__ uint32_t fw_ld(const uint32_t* __restrict__ Mg, uint32_t off /* bytes */) {
  return __ldg(reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(Mg) + off));
}

template <int C>
struct FwVec { uint32_t v[C]; };
template <int C>
__device__ __forceinline__ FwVec<C> fw_load(const uint32_t* p) {
  FwVec<C> o;
  if (C == 2) { const uint2 t = *reinterpret_cast<const uint2*>(p); o.v[0] = t.x; o.v[C - 1] = t.y; }
  else o.v[0] = p[0];
  return o;
}
template <int C>
__device__ __forceinline__ void fw_store(uint32_t* p, const FwVec<C>& o) {
  if (C == 2) *reinterpret_cast<uint2*>(p) = make_uint2(o.v[0], o.v[C - 1]);
  else p[0] = o.v[0];
}

template <int C>
__global__ void __launch_bounds__(kFwMaxWarps * 32, 1) factor_wide_kernel(const FsParams P, const uint32_t* __restrict__ Mg /* r x 32 C, times R^2 */,
                                                                      const uint32_t* __restrict__ rownnz_g, unsigned long long lo,
                                                                      unsigned long long hi, Key* __restrict__ block_best,
                                                                      uint32_t* __restrict__ table /* 3 x (hi-lo) or null */) {
  constexpr unsigned kFull = 0xffffffffu;
  constexpr uint32_t kRowBytes = 32u * C * 4u;
  extern __shared__ __align__(16) uint32_t fw_smem[];
  __shared__ Key red[kFwMaxWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  uint32_t* nnzsh = fw_smem;
  uint32_t* Rw = fw_smem + fw_fixed_words(P.r) + (size_t)warp * fw_warp_words(P.r, P.n, C);  // R[i][lane][c]
  uint32_t* Tw = Rw + (size_t)P.n * 32 * C;                                                           // T[i][lane][c]
  uint32_t* pcw = Tw + (size_t)P.n * 32 * C;  // byte offset of pivot column i inside a row of M
  uint16_t* perm = reinterpret_cast<uint16_t*>(pcw + P.n);
  for (int e = threadIdx.x; e < P.r; e += blockDim.x) nnzsh[e] = rownnz_g[e];
  __syncthreads();
  uint32_t* Rl = Rw + lane * C;
  uint32_t* Tl = Tw + lane * C;

  Key best;
  best.primary = ~0ull; best.index = ~0ull;
  const unsigned long long step = (unsigned long long)gridDim.x * nwarps;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * nwarps + warp; idx < hi; idx += step) {  // warp-uniform
    // ---- row order: Fisher-Yates from the digit stream (every lane computes the digits, lane 0 swaps) ----
    for (int t = lane; t < P.r; t += 32) perm[t] = (uint16_t)t;
    __syncwarp();
    {
      FsDigits ds(P.seed, idx);
      for (int i = 0; i + 1 < P.r; ++i) {
        const uint32_t d = ds.digit((uint32_t)(P.r - i));
        if (lane == 0 && d) { const uint16_t a = perm[i]; perm[i] = perm[i + d]; perm[i + d] = a; }
      }
    }
    __syncwarp();
    // ---- selection pass: R[i][.] = -S R_i, T[i][.] = -S T_i as in factor_sweep_kernel, rows i < nb valid ----
    int nb = 0;
    uint32_t S = P.one;
    for (int t = 0; t < P.r && nb < P.n; ++t) {
      const uint32_t rowo = (uint32_t)perm[t] * kRowBytes;
      FsAcc ar[C], at[C];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        ar[c].lo = 0; ar[c].hi = 0; at[c].lo = 0; at[c].hi = 0;
        fs_mac(ar[c], S, fw_ld(Mg, rowo + 4u * (uint32_t)(lane + 32 * c)));  // S v
        fs_mac(at[c], S, lane + 32 * c == nb ? P.one2 : 0u);                              // S e_nb
      }
      for (int i = 0; i < nb; ++i) {
        const uint32_t cv = fw_ld(Mg, rowo + pcw[i]);  // v[pivot column i]: broadcast
        const FwVec<C> rv = fw_load<C>(Rl + (size_t)i * 32 * C), tv = fw_load<C>(Tl + (size_t)i * 32 * C);
#pragma unroll
        for (int c = 0; c < C; ++c) { fs_mac(ar[c], cv, rv.v[c]); fs_mac(at[c], cv, tv.v[c]); }
      }
      uint32_t vr[C];
      int pcn = -1;  // pivot: the first non-zero coordinate
#pragma unroll
      for (int c = C - 1; c >= 0; --c) {
        vr[c] = fs_reduce(ar[c], P);
        const unsigned m = __ballot_sync(kFull, vr[c] != 0);
        if (m) pcn = 32 * c + __ffs(m) - 1;
      }
      if (pcn < 0) continue;  // dependent on the rows kept so far
      const int ph = pcn >> 5, pl = pcn & 31;
      uint32_t nvr[C], nvt[C];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const uint32_t vt = fs_reduce(at[c], P);
        nvr[c] = vr[c] ? P.p - vr[c] : 0u;
        nvt[c] = vt ? P.p - vt : 0u;
      }
      const uint32_t pv = __shfl_sync(kFull, ph ? vr[C - 1] : vr[0], pl);  // S pv
      for (int i = 0; i < nb; ++i) {
        FwVec<C> rv = fw_load<C>(Rl + (size_t)i * 32 * C), tv = fw_load<C>(Tl + (size_t)i * 32 * C);
        const uint32_t f = __shfl_sync(kFull, ph ? rv.v[C - 1] : rv.v[0], pl);  // -S R_i[pivot column]
#pragma unroll
        for (int c = 0; c < C; ++c) {
          rv.v[c] = mont_mul2(pv, rv.v[c], f, nvr[c], P.p, P.pinv);
          tv.v[c] = mont_mul2(pv, tv.v[c], f, nvt[c], P.p, P.pinv);
        }
        fw_store<C>(Rl + (size_t)i * 32 * C, rv);
        fw_store<C>(Tl + (size_t)i * 32 * C, tv);
      }
      FwVec<C> nr, nt;
#pragma unroll
      for (int c = 0; c < C; ++c) { nr.v[c] = mont_mul(S, nvr[c], P.p, P.pinv); nt.v[c] = mont_mul(S, nvt[c], P.p, P.pinv); }
      fw_store<C>(Rl + (size_t)nb * 32 * C, nr);
      fw_store<C>(Tl + (size_t)nb * 32 * C, nt);
      if (lane == 0) {
        pcw[nb] = 4u * (uint32_t)pcn;
        if (t != nb) { const uint16_t a = perm[nb]; perm[nb] = perm[t]; perm[t] = a; }  // :793-796
      }
      S = mont_mul(S, pv, P.p, P.pinv);
      ++nb;
      __syncwarp();
    }
    // ---- score: the rows outside CoB two at a time, so that each T row loaded serves two of them ----
    const bool ok = nb == P.n;
    uint32_t nnz_alt = 0, nno_alt = 0, nnz_cob = 0;
    if (ok) {
      nnz_alt = (uint32_t)P.k;  // identity rows of Res
      for (int t = 0; t < P.k; ++t) nnz_cob += nnzsh[perm[t]];
      for (int t = P.k; t < P.r; t += 2) {
        const bool two = t + 1 < P.r;
        const uint32_t row0 = (uint32_t)perm[t] * kRowBytes, row1 = two ? (uint32_t)perm[t + 1] * kRowBytes : row0;
        FsAcc a0[C], a1[C];
#pragma unroll
        for (int c = 0; c < C; ++c) { a0[c].lo = 0; a0[c].hi = 0; a1[c].lo = 0; a1[c].hi = 0; }
        for (int i = 0; i < P.n; ++i) {
          const uint32_t pci = pcw[i];
          const uint32_t c0 = fw_ld(Mg, row0 + pci), c1 = fw_ld(Mg, row1 + pci);
          const FwVec<C> tv = fw_load<C>(Tl + (size_t)i * 32 * C);
#pragma unroll
          for (int c = 0; c < C; ++c) { fs_mac(a0[c], c0, tv.v[c]); fs_mac(a1[c], c1, tv.v[c]); }
        }
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const bool col = lane + 32 * c < P.n;
          const uint32_t x0 = fs_reduce(a0[c], P), x1 = fs_reduce(a1[c], P);  // -S times the coordinates
          const bool nz0 = col && x0 != 0, nz1 = two && col && x1 != 0;
          nnz_alt += __popc(__ballot_sync(kFull, nz0)) + __popc(__ballot_sync(kFull, nz1));
          nno_alt += __popc(__ballot_sync(kFull, nz0 && x0 != S && x0 != P.p - S)) + __popc(__ballot_sync(kFull, nz1 && x1 != S && x1 != P.p - S));
        }
      }
    }
    const unsigned long long key = ok ? fs_pack(nnz_alt, nno_alt, nnz_cob) : ~0ull;
    if (table && lane == 0) {
      const unsigned long long o = (idx - lo) * 3;
      table[o] = ok ? nnz_alt : 0xffffffffu; table[o + 1] = ok ? nno_alt : 0u; table[o + 2] = ok ? nnz_cob : 0u;
    }
    if (key < best.primary || (key == best.primary && idx < best.index)) { best.primary = key; best.index = idx; }
    __syncwarp();
  }
  if (lane == 0) red[warp] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    Key b = red[0];
    for (int w = 1; w < nwarps; ++w) if (key_less(red[w], b)) b = red[w];
    block_best[blockIdx.x] = b;
  }
}

typedef void (*FsLaunch)(int grid, int threads, size_t smem, cudaStream_t st, const FsParams& P, const uint32_t* M, const uint32_t* nnz,
                         unsigned long long lo, unsigned long long hi, Key* bb, uint32_t* table);
template <int N>
struct FsWidth { static constexpr int value = N <= 4 ? 4 : N <= 8 ? 8 : N <= 16 ? 16 : 32; };
template <int N>
static void fs_launch(int grid, int threads, size_t smem, cudaStream_t st, const FsParams& P, const uint32_t* M, const uint32_t* nnz,
                      unsigned long long lo, unsigned long long hi, Key* bb, uint32_t* table) {
  factor_sweep_kernel<N, FsWidth<N>::value><<<grid, threads, smem, st>>>(P, M, nnz, lo, hi, bb, table);
}
template <int C>
static void fw_launch(int grid, int threads, size_t smem, cudaStream_t st, const FsParams& P, const uint32_t* M, const uint32_t* nnz,
                      unsigned long long lo, unsigned long long hi, Key* bb, uint32_t* table) {
  factor_wide_kernel<C><<<grid, threads, smem, st>>>(P, M, nnz, lo, hi, bb, table);
}
template <int N>
static int fs_blocks_per_sm(size_t smem) {
  int nb = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, factor_sweep_kernel<N, FsWidth<N>::value>, kFsThreads, smem);
  return nb > 0 ? nb : 1;
}
template <int C>
static cudaError_t fw_blocks_per_sm(int threads, size_t smem, int* bps) {
  const cudaError_t e = cudaFuncSetAttribute(factor_wide_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  *bps = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, factor_wide_kernel<C>, threads, smem);
  if (*bps < 1) *bps = 1;
  return cudaSuccess;
}

static uint32_t host_to_mont(uint64_t a, uint32_t p) { return (uint32_t)((((unsigned __int128)a) << 32) % p); }
static uint32_t host_to_mont2(uint64_t a, uint32_t p) { return (uint32_t)((((unsigned __int128)(a % p)) << 64) % p); }  // a R^2 mod p

}  // namespace plo

using namespace plo;

struct plo_factor_plan {
  FsParams P;
  int grid, threads, per_block;  // per_block: candidates in flight per block
  size_t smem;
  FsLaunch launch;
  char kernel[48];
  uint32_t *d_M, *d_nnz;
  Key* d_bb;
};

extern "C" {

void plo_factor_plan_destroy(plo_factor_plan* pl) {
  if (!pl) return;
  pool_free(pl->d_M); pool_free(pl->d_nnz); pool_free(pl->d_bb);
  delete pl;
}

int plo_factor_plan_create(plo_factor_plan** plan, uint32_t p, int r, int n, int k, const uint32_t* M, uint64_t seed) {
  if (!plan || !M || r < 1 || n < 1 || n > kFwMaxCols || r > kFwMaxRows || k < n || k > r || p < 3 || !(p & 1u) || p >= (1u << 31)) {
    set_error("plo_factor_plan_create: need 1 <= n <= %d, n <= k <= r <= %d, odd prime 3 <= p < 2^31", kFwMaxCols, kFwMaxRows);
    return PLO_E_ARG;
  }
  for (size_t e = 0; e < (size_t)r * n; ++e)
    if (M[e] >= p) { set_error("plo_factor_plan_create: residue >= p"); return PLO_E_ARG; }
  int rc = check_device();
  if (rc) return rc;
  plo_factor_plan* pl = new plo_factor_plan();
  memset(pl, 0, sizeof(*pl));
  FsParams& P = pl->P;
  P.p = p; P.r = r; P.n = n; P.k = k; P.seed = seed; P.M64 = ~0ull / p;
  uint32_t inv = 1;  // Newton: p * inv == 1 mod 2^32
  for (int i = 0; i < 5; ++i) inv *= 2u - p * inv;
  P.pinv = 0u - inv;
  P.one = host_to_mont(1, p); P.one2 = host_to_mont2(1, p);
  // n <= 32 and r < 256: factor_sweep_kernel<N> (register basis, byte row order); every other shape: factor_wide_kernel
  const bool wide = n > 32 || r > kFsMaxRows - 1;
  const int C = n > 32 ? 2 : 1;  // columns per lane of the wide kernel; M is stored r x 32 C
  std::vector<uint32_t> hM((size_t)r * 32 * C, 0), hn(r, 0);
  for (int i = 0; i < r; ++i)
    for (int j = 0; j < n; ++j) { hM[(size_t)i * 32 * C + j] = host_to_mont2(M[(size_t)i * n + j], p); hn[i] += M[(size_t)i * n + j] != 0; }
  int bps = 1;
  if (!wide) {
    const int npad = (n + 3) & ~3;
    switch (npad) {
#define PLO_FS_CASE(NN) case NN: pl->launch = &fs_launch<NN>; break;
      PLO_FS_CASE(4) PLO_FS_CASE(8) PLO_FS_CASE(12) PLO_FS_CASE(16) PLO_FS_CASE(20) PLO_FS_CASE(24) PLO_FS_CASE(28) PLO_FS_CASE(32)
#undef PLO_FS_CASE
    }
    snprintf(pl->kernel, sizeof(pl->kernel), "factor_sweep_kernel<%d>", npad);
    const int width = npad <= 4 ? 4 : npad <= 8 ? 8 : npad <= 16 ? 16 : 32;  // lanes per candidate
    const int group = 32 / width;
    pl->threads = kFsThreads;
    pl->per_block = kFsWarps * group;
    pl->smem = ((size_t)r * kFsStride + r) * 4 + (size_t)kFsWarps * group * kFsMaxRows;
    switch (npad) {
#define PLO_FS_CASE(NN) case NN: bps = fs_blocks_per_sm<NN>(pl->smem); break;
      PLO_FS_CASE(4) PLO_FS_CASE(8) PLO_FS_CASE(12) PLO_FS_CASE(16) PLO_FS_CASE(20) PLO_FS_CASE(24) PLO_FS_CASE(28) PLO_FS_CASE(32)
#undef PLO_FS_CASE
    }
  } else {
    // one block per SM with as many warps as its shared memory holds, at most kFwMaxWarps
    int dev = 0, optin = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaFuncAttributes fa;
    const cudaError_t fe = cudaFuncGetAttributes(&fa, C == 1 ? (const void*)factor_wide_kernel<1> : (const void*)factor_wide_kernel<2>);
    if (fe != cudaSuccess) { set_error("plo_factor_plan_create: %s", cudaGetErrorString(fe)); plo_factor_plan_destroy(pl); return PLO_E_CUDA; }
    const size_t ww = fw_warp_words(r, n, C) * 4, fix = fw_fixed_words(r) * 4;
    const size_t avail = (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : 0;  // the dynamic share: optin minus the static red[]
    const int warps = (int)std::min<size_t>(kFwMaxWarps, avail > fix ? (avail - fix) / ww : 0);
    if (warps < 1) { set_error("plo_factor_plan_create: %d x %d needs more shared memory than a block has", r, n); plo_factor_plan_destroy(pl); return PLO_E_ARG; }
    pl->threads = warps * 32;
    pl->per_block = warps;
    pl->smem = fix + (size_t)warps * ww;
    cudaError_t e;
    if (C == 1) { pl->launch = &fw_launch<1>; e = fw_blocks_per_sm<1>(pl->threads, pl->smem, &bps); }
    else { pl->launch = &fw_launch<2>; e = fw_blocks_per_sm<2>(pl->threads, pl->smem, &bps); }
    if (e != cudaSuccess) { set_error("plo_factor_plan_create: %s", cudaGetErrorString(e)); plo_factor_plan_destroy(pl); return PLO_E_CUDA; }
    snprintf(pl->kernel, sizeof(pl->kernel), "factor_wide_kernel<%d>", C);
  }
  pl->grid = sm_count() * bps;
  const bool ok = pool_alloc(&pl->d_M, hM.size() * 4) == cudaSuccess && pool_alloc(&pl->d_nnz, hn.size() * 4) == cudaSuccess &&
                  pool_alloc(&pl->d_bb, sizeof(Key) * pl->grid) == cudaSuccess &&
                  cudaMemcpy(pl->d_M, hM.data(), hM.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
                  cudaMemcpy(pl->d_nnz, hn.data(), hn.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok) { set_error("plo_factor_plan_create: %s", cudaGetErrorString(cudaGetLastError())); plo_factor_plan_destroy(pl); return PLO_E_CUDA; }
  *plan = pl;
  return PLO_OK;
}

static int fs_grid(const plo_factor_plan* pl, uint64_t lo, uint64_t hi) {
  const uint64_t per_block = (uint64_t)pl->per_block;
  const uint64_t need = (hi - lo + per_block - 1) / per_block;
  return (int)(need < (uint64_t)pl->grid ? (need ? need : 1) : (uint64_t)pl->grid);
}

int plo_factor_plan_run(plo_factor_plan* pl, uint64_t lo, uint64_t hi, void* stream) {
  if (!pl) { set_error("plo_factor_plan_run: null plan"); return PLO_E_ARG; }
  const int grid = fs_grid(pl, lo, hi);
  Key none;
  none.primary = ~0ull; none.index = ~0ull;
  std::vector<Key> init(pl->grid, none);
  PLO_CUDA(cudaMemcpyAsync(pl->d_bb, init.data(), sizeof(Key) * pl->grid, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  if (hi > lo) pl->launch(grid, pl->threads, pl->smem, (cudaStream_t)stream, pl->P, pl->d_M, pl->d_nnz, lo, hi, pl->d_bb, nullptr);
  PLO_CUDA(cudaGetLastError());
  return PLO_OK;
}

int plo_factor_plan_result(plo_factor_plan* pl, void* stream, plo_factor_best* best) {
  if (!pl || !best) { set_error("plo_factor_plan_result: bad argument"); return PLO_E_ARG; }
  std::vector<Key> bb(pl->grid);
  PLO_CUDA(cudaMemcpyAsync(bb.data(), pl->d_bb, sizeof(Key) * pl->grid, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  PLO_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  Key b = bb[0];
  for (const Key& x : bb) if (key_less(x, b)) b = x;
  best->index = b.index;
  if (b.primary == ~0ull) { best->nnz_alt = best->nno_alt = best->nnz_cob = 0xffffffffu; best->index = PLO_NO_INDEX; }
  else { best->nnz_alt = (uint32_t)(b.primary >> 40); best->nno_alt = (uint32_t)((b.primary >> 20) & 0xfffffu); best->nnz_cob = (uint32_t)(b.primary & 0xfffffu); }
  return PLO_OK;
}

int plo_factor_plan_launches(const plo_factor_plan*) { return 1; }

int plo_factor_plan_kernel(const plo_factor_plan* pl, char* name, int cap) {
  if (!pl || !name || cap < 1) { set_error("plo_factor_plan_kernel: bad argument"); return PLO_E_ARG; }
  snprintf(name, (size_t)cap, "%s", pl->kernel);
  return PLO_OK;
}

int plo_factor_sweep(uint32_t p, int r, int n, int k, const uint32_t* M, uint64_t seed, uint64_t lo, uint64_t hi,
                     plo_factor_best* best, uint32_t* table) {
  plo_factor_plan* pl = nullptr;
  int rc = plo_factor_plan_create(&pl, p, r, n, k, M, seed);
  if (rc) return rc;
  if (!table) {
    rc = plo_factor_plan_run(pl, lo, hi, nullptr);
  } else {
    uint32_t* d_tab = nullptr;
    const size_t cnt = (size_t)(hi > lo ? hi - lo : 0) * 3;
    Key none;
    none.primary = ~0ull; none.index = ~0ull;
    std::vector<Key> init(pl->grid, none);
    if (cudaMemcpy(pl->d_bb, init.data(), sizeof(Key) * pl->grid, cudaMemcpyHostToDevice) != cudaSuccess ||
        pool_alloc(&d_tab, cnt ? cnt * 4 : 4) != cudaSuccess) {
      set_error("plo_factor_sweep: %s", cudaGetErrorString(cudaGetLastError())); plo_factor_plan_destroy(pl); return PLO_E_CUDA;
    }
    if (hi > lo) pl->launch(fs_grid(pl, lo, hi), pl->threads, pl->smem, nullptr, pl->P, pl->d_M, pl->d_nnz, lo, hi, pl->d_bb, d_tab);
    if (cudaMemcpy(table, d_tab, cnt * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_error("plo_factor_sweep: %s", cudaGetErrorString(cudaGetLastError())); rc = PLO_E_CUDA; }
    pool_free(d_tab);
  }
  if (!rc && best) rc = plo_factor_plan_result(pl, nullptr, best);
  plo_factor_plan_destroy(pl);
  return rc;
}

// Row order of candidate `index`: perm[t] = original row at position t (before the selection swaps).
int plo_factor_decode(int r, uint64_t seed, uint64_t index, int32_t* perm) {
  if (r < 1 || !perm) { set_error("plo_factor_decode: bad argument"); return PLO_E_ARG; }
  for (int t = 0; t < r; ++t) perm[t] = t;
  FsDigits ds(seed, index);
  for (int i = 0; i + 1 < r; ++i) {
    const uint32_t d = ds.digit((uint32_t)(r - i));
    std::swap(perm[i], perm[i + d]);
  }
  return PLO_OK;
}

}  // extern "C"
