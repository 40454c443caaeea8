// lincomb_quad.cu -- ALL the rows of one inner block of localSparsifier in one launch sequence
// ("score once, filter four times").
//
// Reference: include/plinopt_sparsify.inl:282-326.  For one inner block (positions off..off+3 of the candidate vector) the
// reference runs the quad loop (:299-314) once per row num = 0..3; the score (rlHw, clHw) of a candidate (:176-180) does not
// depend on num -- only the independence filter rank(Cand) > num (:172-175) and the weight seed (:290-295) do.  So:
//
//   quad_tables_kernel   product tables C_l . TM[off+t][.] in the field, built on the device from TM and Coeffs
//   quad_count_kernel    zero count rl of EVERY candidate, once (same prefix/compare formulation as lincomb_kernel), one byte each
//   quad_pick_kernel x4  row num: keep-best over the stored counts with the independence filter against the rows chosen so far.
//                        The annihilator functionals of step num are rebuilt by thread 0 of every block from the winners of the
//                        previous picks (minors of their images under the initial functionals): no host round trip between rows.
//
// One host->device copy (descriptors + TM + Coeffs), six launches (ten with two-phase picks), one device->host copy per call, for any number of independent
// problems (the column blocks of blockSparsifier, :710-723, advance in lock step).  Winners are bit-identical to four successive
// plo_lincomb_search calls (tests/test_gpu_lincomb.py).
#include <cstring>

#include "lincomb_common.cuh"

namespace plo {

struct QuadDesc {  // one problem; built on the host, read by every kernel
  int n, m, c, nact;             // nact = live positions = rows to choose = min(4, n - off)
  int mpad, cl_const, nphi0, seed_mode;
  int lsplit, npick;             // npick = rows this call decides = nact - (rows of this block already among the previous rows)
  unsigned int p, pad1;
  unsigned long long tab_off;    // element offset of t0 in the table region (t1, t2, t3 follow at + c*mpad each)
  unsigned long long cnt_off;    // byte offset of the c^4 zero counts (16-byte aligned), followed by the c^3 per-prefix maxima
  unsigned long long in_off;     // int64 offset of [TM live rows: 4 x m | coef: c] in the staging buffer
  unsigned long long zf_off;     // byte offset of zflag[4][c]
  unsigned long long seed_key;   // weight seed of the first row
  long long cmax;                // max |coef| (exact path: magnitude guard of the functionals)
  unsigned long long m64;        // floor((2^64 - 1) / p) for the Barrett reductions (p > 0)
  unsigned long long inv_off;    // 32-bit word offset of this problem's inverse-lookup tables (mod p, c >= 32)
  int hbits, pad2;
  long long phi0[16];            // annihilator functionals of the rows known before this call, on the live positions
  long long seedvec[4];          // the vector holding the seed weight, on the live positions (seed_mode == 1)
};

constexpr int kPickThreads = 256;

// ---- tables -----------------------------------------------------------------------------------------------------------
template <typename T, bool MODP>
__global__ void __launch_bounds__(256) quad_tables_kernel(const QuadDesc* __restrict__ descs, const long long* __restrict__ stage, T* __restrict__ tables,
                                                           unsigned char* __restrict__ zflags, unsigned long long* __restrict__ results, int* __restrict__ status,
                                                           const unsigned int* __restrict__ invtabs /* inverse-lookup path: T0..T2 are stored times -A3_e^-1, else NULL */) {
  const QuadDesc& d = descs[blockIdx.y];
  const int c = d.c, m = d.m, mpad = d.mpad, nact = d.nact;
  const long long* __restrict__ tm = stage + d.in_off;       // [4][m]
  const long long* __restrict__ coef = tm + 4 * (size_t)m;   // [c]
  const size_t tab = (size_t)c * mpad;
  T* __restrict__ t0 = tables + d.tab_off;
  const size_t total = 4 * tab;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int t = (int)(e / tab);
    const size_t rem = e - (size_t)t * tab;
    const int l = (int)(rem / mpad), j = (int)(rem - (size_t)l * mpad);
    T val = 0;
    if (t < nact && j < m) {
      if (MODP) {
        val = (T)(((unsigned long long)coef[l] * (unsigned long long)tm[(size_t)t * m + j]) % d.p);
        if (invtabs && t < 3) {
          const unsigned int ni = invtabs[d.inv_off + j];
          if (ni != InvTables::kEmpty) val = (T)(((unsigned long long)val * ni) % d.p);
        }
      } else val = (T)(coef[l] * tm[(size_t)t * m + j]);
    }
    if (t == 2) t0[2 * tab + (size_t)j * c + l] = val;  // transposed: consecutive k coalesce in the count kernel
    else t0[(size_t)t * tab + rem] = val;
  }
  if (blockIdx.x == 0) {
    unsigned char* zf = zflags + d.zf_off;
    for (int e = threadIdx.x; e < 4 * c; e += blockDim.x) zf[e] = (e / c < nact) && (coef[e % c] == 0);
    if (threadIdx.x < 4) results[blockIdx.y * 4 + threadIdx.x] = threadIdx.x == 0 ? d.seed_key : pack_key(-1, -1, kIdxMask);
    if (threadIdx.x == 0) status[blockIdx.y] = 0;
  }
}

// ---- zero counts of every candidate, once --------------------------------------------------------------------------------
template <typename T, int MPAD, bool MODP>
__global__ void __launch_bounds__(kLcThreads) quad_count_kernel(const QuadDesc* __restrict__ descs, const T* __restrict__ tables, unsigned char* __restrict__ counts, int max_rows) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* t3s = reinterpret_cast<T*>(smem_raw);
  constexpr int VEC = 16 / sizeof(T);
  const QuadDesc& d = descs[blockIdx.y];
  const int c = d.c, lsplit = d.lsplit;
  const unsigned int p = d.p;
  const size_t tab = (size_t)c * MPAD;
  const T* __restrict__ t0 = tables + d.tab_off;
  const T* __restrict__ t1 = t0 + tab;
  const T* __restrict__ t2 = t1 + tab;
  const T* __restrict__ t3 = t2 + tab;
  unsigned char* __restrict__ cnt = counts + d.cnt_off;
  unsigned char* __restrict__ rmax = cnt + ((size_t)c * c * c * c + 15) / 16 * 16;
  const unsigned long long nitems = (unsigned long long)c * c * c * (unsigned)lsplit;
  const unsigned long long nthreads = (unsigned long long)gridDim.x * kLcThreads;
  if ((unsigned long long)blockIdx.x * kLcThreads >= nitems) return;
  const int ltile = c < max_rows ? c : max_rows;
  for (int l0 = 0; l0 < c; l0 += ltile) {
    const int l1 = min(c, l0 + ltile);
    __syncthreads();
    {
      const uint4* src = reinterpret_cast<const uint4*>(t3 + (size_t)l0 * MPAD);
      uint4* dst = reinterpret_cast<uint4*>(t3s);
      const int nvec = (l1 - l0) * MPAD / VEC;
      for (int e = threadIdx.x; e < nvec; e += kLcThreads) dst[e] = src[e];
    }
    __syncthreads();
    const int lc = (l1 - l0 + lsplit - 1) / lsplit;
    for (unsigned long long item = (unsigned long long)blockIdx.x * kLcThreads + threadIdx.x; item < nitems; item += nthreads) {
      const unsigned long long q = item / (unsigned)lsplit;
      const int s = (int)(item - q * (unsigned)lsplit);
      const int la = l0 + s * lc, lb = min(l1, la + lc);
      if (la >= lb) continue;
      int i, j, k;
      decode_prefix(q, c, i, j, k);
      T nb[MPAD];
#pragma unroll
      for (int e = 0; e < MPAD; ++e) {
        const T a0 = t0[(size_t)i * MPAD + e], a1 = t1[(size_t)j * MPAD + e], a2 = t2[(size_t)e * c + k];
        nb[e] = neg_prefix_sum<T, MODP>(a0, a1, a2, p);
        if (e >= d.m) nb[e] = pad_sentinel<T, MODP>();
      }
      unsigned char* out = cnt + q * (unsigned)c;
      int rowmax = 0;
      for (int l = la; l < lb; ++l) {
        const int rl = zero_count(t3s + (size_t)(l - l0) * MPAD, nb);
        out[l] = (unsigned char)rl;
        rowmax = max(rowmax, rl);
      }
      // largest count of the prefix row: lets the picks skip whole rows.  A row shared by several threads (l range split, or T3 in
      // several tiles) gets the conservative 255.
      if (lsplit == 1 && ltile >= c) rmax[q] = (unsigned char)rowmax; else if (s == 0 && l0 == 0) rmax[q] = 255;
    }
  }
}

// ---- the same counts by inverse lookup (mod p, many coefficients; lincomb_common.cuh "inverse lookup") ---------------------------
// One hash probe per coordinate instead of c compares; the c byte counters of a prefix are built in shared memory and stored as words.
template <int MPAD>
__global__ void __launch_bounds__(kLcThreads) quad_count_inv_kernel(const QuadDesc* __restrict__ descs, const unsigned int* __restrict__ tables,
                                                                    const unsigned int* __restrict__ invtabs, unsigned char* __restrict__ counts,
                                                                    unsigned int* __restrict__ rhist) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned int sh_hist[256];  // how many prefix rows of this block have which largest count
  const QuadDesc& d = descs[blockIdx.y];
  const int c = d.c, hsize = 1 << d.hbits, cpad = (c + 3) & ~3;
  const unsigned int p = d.p;
  const unsigned nprefix = (unsigned)c * c * c;
  if ((unsigned long long)blockIdx.x * kLcThreads >= nprefix) return;
  unsigned int* ninv = reinterpret_cast<unsigned int*>(smem_raw);
  uint2* htab = reinterpret_cast<uint2*>(ninv + MPAD);
  unsigned int* nextdup = reinterpret_cast<unsigned int*>(htab + hsize);
  unsigned char* hist = reinterpret_cast<unsigned char*>(nextdup + c) + (size_t)threadIdx.x * (cpad + 4);
  for (int e = threadIdx.x; e < 256; e += kLcThreads) sh_hist[e] = 0u;
  {
    const unsigned int* src = invtabs + d.inv_off;
    const int nw = (int)InvTables::words(MPAD, hsize, c);
    for (int e = threadIdx.x; e < nw; e += kLcThreads) ninv[e] = src[e];
  }
  __syncthreads();
  const InvShared sh = inv_shared_addresses(ninv, htab, nextdup, hist);
  const size_t tab = (size_t)c * MPAD;
  const unsigned int* __restrict__ t0 = tables + d.tab_off;
  const unsigned int* __restrict__ t1 = t0 + tab;
  const unsigned int* __restrict__ t2 = t1 + tab;
  unsigned char* __restrict__ cnt = counts + d.cnt_off;
  unsigned char* __restrict__ rmax = cnt + ((size_t)c * c * c * c + 15) / 16 * 16;
  const bool words_ok = (c & 3) == 0;
  const int lane = threadIdx.x & 31, hstride = cpad + 4;
  const unsigned char* hist_w = hist - (size_t)lane * hstride;  // counters of lane 0 of this warp
  // The 32 prefixes of a warp are consecutive, so their c counts each form ONE contiguous block of 32 c bytes: the warp stores it
  // together, lane after lane along the block (coalesced 128 B stores; a thread storing its own row word by word costs 32 sectors
  // per store instruction).
  for (unsigned q0 = blockIdx.x * kLcThreads + (threadIdx.x - lane); q0 < nprefix; q0 += gridDim.x * kLcThreads) {
    const unsigned q = q0 + lane;
    const bool valid = q < nprefix;
    unsigned base = 0, mx = 0;  // coordinates that vanish for every l; per-byte maximum of the hit counters
    if (valid) {
      int i, j, k;
      decode_prefix(q, c, i, j, k);
      for (int w = 0; w < cpad; w += 4) *reinterpret_cast<unsigned int*>(hist + w) = 0u;
      base = inv_count_prefix(t0 + (size_t)i * MPAD, t1 + (size_t)j * MPAD, t2 + k, c, d.m, p, d.hbits, sh);
    }
    if (words_ok) {
      if (valid) {
        for (int w = 0; w < c; w += 4) mx = __vmaxu4(mx, *reinterpret_cast<const unsigned int*>(hist + w));
      }
      __syncwarp();
      const unsigned rows = min(32u, nprefix - q0), wpr = (unsigned)c >> 2, total = rows * wpr;  // words per row, words of the warp's block
      unsigned int* outw = reinterpret_cast<unsigned int*>(cnt + (size_t)q0 * c);
      for (unsigned idx = lane; idx < ((total + 31u) & ~31u); idx += 32) {
        const unsigned r = min(idx / wpr, rows - 1u), w = idx - (idx / wpr) * wpr;
        const unsigned add = __shfl_sync(0xffffffffu, base, (int)r) * 0x01010101u;  // counts stay below 256: at most m <= 64 per candidate
        if (idx < total) outw[idx] = *reinterpret_cast<const unsigned int*>(hist_w + (size_t)r * hstride + 4u * w) + add;
      }
      __syncwarp();
    } else if (valid) {
      unsigned char* out = cnt + (size_t)q * c;
      for (int l = 0; l < c; ++l) { mx = max(mx, (unsigned)hist[l]); out[l] = (unsigned char)(hist[l] + base); }
    }
    if (valid) {
      mx = max(max(mx & 0xFFu, (mx >> 8) & 0xFFu), max((mx >> 16) & 0xFFu, mx >> 24));
      rmax[q] = (unsigned char)(base + mx);  // largest count of the prefix row: lets the picks skip whole rows
      atomicAdd(&sh_hist[(base + mx) & 0xFFu], 1u);
    }
  }
  __syncthreads();
  if (rhist)  // per problem: the picks start from the level the best rows are at instead of climbing there
    for (int e = threadIdx.x; e < 256; e += kLcThreads) if (sh_hist[e]) atomicAdd(rhist + (size_t)blockIdx.y * 256 + e, sh_hist[e]);
}

// ---- annihilator functionals of step `num` from the winners of the previous picks --------------------------------------------
// Psi (nphi0 x 4) annihilates the rows known before the call; for vectors supported on the live positions, w is in
// span(known rows, w_0..w_{t-1}) iff Psi.w is in span(Psi.w_0, .., Psi.w_{t-1}) =: span(u_0..u_{t-1}) inside F^q (q = nphi0).
// A spanning set of the functionals on F^q that vanish on u_0..u_{t-1} is written down with minors (no division, no growth
// beyond degree t in the u's) and composed with Psi.
__device__ __forceinline__ void ring_init(DevField<false>& R, const QuadDesc& d) { R.p = d.p; }
__device__ __forceinline__ void ring_init(DevField<true>& R, const QuadDesc& d) { R.p = d.p; R.m64 = d.m64; }

// returns 0 ok, 1 stop (an earlier row has no winner: the host takes over), 3 magnitude guard.
// Called by ALL 32 lanes of warp 0 while the rest of the block waits, once per row.  The work is a few hundred dependent modular /
// 128-bit multiply-adds; on one thread that is ~20 us of pure latency, so every stage is spread over the lanes (one output per
// lane, rolled code, a small workspace in shared memory).  Spanning sets with a fixed shape replace pivoting (functionals that
// come out as zero never witness independence, so padding is harmless):
//   t = 0: e_0..e_3            t = 1: u_a e_b - u_b e_a, a < b (6)
//   t = 2: the cross products of (u_0, u_1) restricted to three coordinates (4)      t = 3: the cross product of u_0, u_1, u_2 (1)
constexpr int kMaxPhi = 6;
constexpr unsigned int kTopRows = 512;  // phase 1 of a pick looks at (at least) this many best prefix rows
constexpr int kPrepWords = 16 + 12 + 12 + 6 + 4 * kMaxPhi;  // Psi | winners | u | 2x2 minors | psi
__device__ __forceinline__ int minor_index(int a, int b) { return a == 0 ? b - 1 : (a == 1 ? b + 1 : 5); }  // a < b: 01 02 03 12 13 23

template <bool MODP>
__device__ __noinline__ int quad_prepare(const QuadDesc& d, const long long* __restrict__ coef, const unsigned long long* __restrict__ res, int num,
                                         long long* phi_out, int* nphi_out, typename DevField<MODP>::V* ws) {
  typedef DevField<MODP> Ring;
  typedef typename Ring::V V;
  Ring R;
  ring_init(R, d);
  const int lane = threadIdx.x & 31;
  const int c = d.c;
  V* Psi = ws;        // [4][4]
  V* wv = Psi + 16;   // [3][4] winners of the previous rows on the live positions
  V* u = wv + 12;     // [3][4] their images under Psi
  V* M2 = u + 12;     // [6]
  V* psi = M2 + 6;    // [kMaxPhi][4]
  if (lane < 16) Psi[lane] = R.from((lane >> 2) < d.nphi0 ? d.phi0[lane] : 0);
  bool stop = false;
  if (lane < 3) {
    long long w[4] = {0, 0, 0, 0};
    if (lane < num) {
      const unsigned long long key = res[lane];
      const unsigned long long seed = lane == 0 ? d.seed_key : pack_key(-1, -1, kIdxMask);
      if (key == seed) {
        if (lane == 0 && d.seed_mode == 1) { w[0] = d.seedvec[0]; w[1] = d.seedvec[1]; w[2] = d.seedvec[2]; w[3] = d.seedvec[3]; }
        else stop = true;
      } else {
        int i, j, k, l;
        decode_index(kIdxMask - 1ull - (key & kIdxMask), c, i, j, k, l);
        w[0] = coef[i]; w[1] = d.nact > 1 ? coef[j] : 0; w[2] = d.nact > 2 ? coef[k] : 0; w[3] = d.nact > 3 ? coef[l] : 0;  // Q4: positions beyond n are truncated
      }
    }
    wv[lane * 4 + 0] = R.from(w[0]); wv[lane * 4 + 1] = R.from(w[1]); wv[lane * 4 + 2] = R.from(w[2]); wv[lane * 4 + 3] = R.from(w[3]);
  }
  if (__any_sync(0xffffffffu, stop)) return 1;
  __syncwarp();
  if (lane < 12) {  // u[t][a] = Psi[a] . w_t
    const int t = lane >> 2, a = lane & 3;
    V acc = R.from(0);
#pragma unroll 1
    for (int sx = 0; sx < 4; ++sx) acc = R.add(acc, R.mul(Psi[a * 4 + sx], wv[t * 4 + sx]));
    u[lane] = acc;
  }
  __syncwarp();
  if (lane < 6 && num >= 2) {  // 2x2 minors of (u_0, u_1)
    const int a = lane < 3 ? 0 : (lane < 5 ? 1 : 2), bb = lane < 3 ? lane + 1 : (lane < 5 ? lane - 1 : 3);
    M2[lane] = R.sub(R.mul(u[a], u[4 + bb]), R.mul(u[bb], u[4 + a]));
  }
  __syncwarp();
  const int npsi = num == 0 ? 4 : (num == 1 ? 6 : (num == 2 ? 4 : 1));
  if (lane < 4 * kMaxPhi) {
    const int sfn = lane >> 2, a = lane & 3;
    V val = R.from(0);
    if (num == 0) {
      if (sfn == a) val = R.from(1);
    } else if (num == 1) {
      const int pa = sfn < 3 ? 0 : (sfn < 5 ? 1 : 2), pb = sfn < 3 ? sfn + 1 : (sfn < 5 ? sfn - 1 : 3);
      if (a == pb) val = u[pa];
      else if (a == pa) val = R.neg(u[pb]);
    } else {
      // omitted coordinate dd, remaining x < y < z: (M_yz, -M_xz, M_xy) on (x, y, z); for the last row the same three minors are
      // contracted with u_2 into (-1)^dd det(u_0, u_1, u_2 without column dd)
      const int dd = num == 2 ? sfn : a;
      const int x = dd == 0 ? 1 : 0, y = dd <= 1 ? 2 : 1, z = dd <= 2 ? 3 : 2;
      if (num == 2 && sfn < 4) {
        if (a == x) val = M2[minor_index(y, z)];
        else if (a == y) val = R.neg(M2[minor_index(x, z)]);
        else if (a == z) val = M2[minor_index(x, y)];
      } else if (num == 3 && sfn == 0) {
        const V det = R.add(R.sub(R.mul(u[8 + x], M2[minor_index(y, z)]), R.mul(u[8 + y], M2[minor_index(x, z)])), R.mul(u[8 + z], M2[minor_index(x, y)]));
        val = (dd & 1) ? R.neg(det) : det;
      }
    }
    psi[lane] = val;
  }
  __syncwarp();
  bool over = false;
  if (lane < 4 * npsi) {  // compose with Psi and narrow
    const int sfn = lane >> 2, pos = lane & 3;
    V acc = R.from(0);
#pragma unroll 1
    for (int a = 0; a < 4; ++a) acc = R.add(acc, R.mul(psi[sfn * 4 + a], Psi[a * 4 + pos]));
    if (!MODP) {
      const V lim = (V)((((unsigned long long)1 << 62) - 1) / (unsigned long long)(4 * (d.cmax > 0 ? d.cmax : 1)));
      over = R.magnitude(acc) > lim;
    }
    phi_out[lane] = (long long)acc;
  }
  if (__any_sync(0xffffffffu, over)) return 3;
  if (lane == 0) *nphi_out = npsi;
  return 0;
}

// ---- row `num`: keep-best over the stored counts --------------------------------------------------------------------------------
template <bool MODP>
__global__ void __launch_bounds__(kPickThreads) quad_pick_kernel(const QuadDesc* __restrict__ descs, const long long* __restrict__ stage,
                                                                 const unsigned char* __restrict__ zflags, const unsigned char* __restrict__ counts,
                                                                 unsigned long long* __restrict__ results, int* __restrict__ status, int num,
                                                                 const unsigned int* __restrict__ rhist, int phase) {
  // phase 0: the whole pick.  With the histogram of the row maxima (inverse-lookup path) a pick is two launches: phase 1 looks only at
  // the rows whose largest count is among the kTopRows best -- the maximum over the independent candidates is found there unless every
  // candidate of those rows depends on the rows chosen so far -- and phase 2, the whole pick, returns at once when phase 1 published
  // a winner (a winner with count >= the floor IS the maximum: everything at or above the floor was looked at).
  __shared__ long long sh_phi[4 * kMaxPhi];
  __shared__ int sh_nphi, sh_stop;
  __shared__ unsigned long long red[32];
  __shared__ __align__(16) typename DevField<MODP>::V sh_ws[kPrepWords];
  const int b = blockIdx.y;
  const QuadDesc& d = descs[b];
  if (num >= d.npick) return;
  if (phase == 2 && *reinterpret_cast<volatile unsigned long long*>(results + b * 4 + num) > (num == 0 ? d.seed_key : pack_key(-1, -1, kIdxMask))) return;
  const int c = d.c;
  const unsigned long long N4 = (unsigned long long)c * c * c * c;
  const unsigned long long nchunks = (N4 + 15) / 16;
  if ((unsigned long long)blockIdx.x * kPickThreads >= nchunks) return;
  const long long* __restrict__ coef = stage + d.in_off + 4 * (size_t)d.m;
  if (threadIdx.x < 32) {
    const int rc = quad_prepare<MODP>(d, coef, results + b * 4, num, sh_phi, &sh_nphi, sh_ws);
    if (threadIdx.x == 0) {
      sh_stop = rc;
      if (rc == 3 && blockIdx.x == 0) status[b] = 3;
    }
  }
  __syncthreads();
  if (sh_stop) return;
  const int nphi = sh_nphi;
  const unsigned char* __restrict__ zf = zflags + d.zf_off;
  const uint4* __restrict__ cnt = reinterpret_cast<const uint4*>(counts + d.cnt_off);
  const unsigned long long seed = num == 0 ? d.seed_key : pack_key(-1, -1, kIdxMask);
  unsigned long long best = seed;
  {
    const unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(results + b * 4 + num);  // winners other blocks already published
    if (cur > best) best = cur;
  }
  int best_rl1 = (int)(best >> 48);
  {
    // A thread takes whole prefix rows (c bytes): one index decode per c candidates and a running best that has seen whole rows.
    // The count kernels left the largest count of every row beside the counts (c^3 bytes): a row that cannot reach the best count
    // known to the BLOCK is skipped without being read, so after the first rows a pick reads c^3 bytes instead of c^4.
    // (Tried: reading everything -- thread per row, lane per word of a shared row, rows staged through shared memory: 1.1-1.9 ms
    // per pick at c = 128, latency-bound at ~1 TB/s with the few warps this register-heavy kernel keeps resident.)
    __shared__ int sh_best_rl1;
    if (threadIdx.x == 0) {
      int floor1 = best_rl1;
      if (phase == 1) {
        unsigned int seen = 0;
        int v = 255;
        for (; v > 0; --v) { seen += rhist[(size_t)b * 256 + v]; if (seen >= kTopRows) break; }
        floor1 = max(floor1, v + 1);  // rows whose largest count is below v are not looked at in this phase
      }
      sh_best_rl1 = floor1;
    }
    __syncthreads();
    if (phase == 1) best_rl1 = max(best_rl1, sh_best_rl1);
    const unsigned nprefix = (unsigned)c * c * c;
    const unsigned char* __restrict__ bytes = counts + d.cnt_off;
    const unsigned char* __restrict__ rmax = bytes + (N4 + 15) / 16 * 16;
    const bool words_ok = (c & 3) == 0;
    for (unsigned q = blockIdx.x * kPickThreads + threadIdx.x; q < nprefix; q += gridDim.x * kPickThreads) {
      const int floor_rl1 = max(best_rl1, *reinterpret_cast<volatile int*>(&sh_best_rl1));
      if ((int)rmax[q] + 1 < floor_rl1) continue;
      int i, j, k;
      decode_prefix(q, c, i, j, k);
      const int zc = d.cl_const + zf[i] + zf[c + j] + zf[2 * c + k];
      const unsigned char* row = bytes + (size_t)q * c;
      for (int l0 = 0; l0 < c; l0 += 4) {
        unsigned int w;
        if (words_ok) w = __ldg(reinterpret_cast<const unsigned int*>(row + l0));
        else {
          w = 0;
          for (int t = 0; t < 4 && l0 + t < c; ++t) w |= (unsigned)row[l0 + t] << (8 * t);
        }
        const unsigned thr = (unsigned)(floor_rl1 > 0 ? floor_rl1 - 1 : 0) * 0x01010101u;
        if (__vcmpgeu4(w, thr) == 0u) continue;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int l = l0 + t;
          const int rl = (int)((w >> (8 * t)) & 0xFFu);
          if (l < c && rl + 1 >= best_rl1) {
            const int cl = zc + zf[3 * c + l];
            const unsigned long long idx = (unsigned long long)q * (unsigned)c + (unsigned)l;
            const unsigned long long key = pack_key(rl, cl, kIdxMask - 1ull - idx);
            if (key > best && independent<MODP>(sh_phi, nphi, coef, d.p, d.m64, i, j, k, l)) {
              best = key;
              best_rl1 = rl + 1;
              atomicMax(&sh_best_rl1, best_rl1);
            }
          }
        }
      }
    }
  }
  block_max<kPickThreads>(best, threadIdx.x, red, [&](unsigned long long v) { if (v > seed) atomicMax(results + b * 4 + num, v); });
}

// ---- small searches: everything in ONE launch, one block per problem -----------------------------------------------------------
// For c <= ~20 the four product tables and the c^4 zero counts fit the shared memory of one SM: tables, counts and the picks
// of all rows run inside one block (512 threads), rows separated by __syncthreads instead of kernel boundaries.  This is the path
// of the default `sparsifier -c 11` (c = 3, 7, 11): one copy in, one launch, one copy out per localSparsifier round.
constexpr int kSmallThreads = 512;
__host__ __device__ inline size_t quad_small_smem(int c, int mpad, int width) {
  const size_t n4 = ((size_t)c * c * c * c + 15) / 16 * 16;
  return (size_t)4 * c * mpad * width + n4 + (size_t)8 * c + ((size_t)4 * c + 15) / 16 * 16;
}

template <typename T, int MPAD, bool MODP>
__global__ void __launch_bounds__(kSmallThreads) quad_small_kernel(const QuadDesc* __restrict__ descs, const long long* __restrict__ stage,
                                                                   unsigned long long* __restrict__ results, int* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ long long sh_phi[4 * kMaxPhi];
  __shared__ int sh_nphi, sh_stop;
  __shared__ unsigned long long red[32], sh_res[4], sh_best;
  __shared__ __align__(16) typename DevField<MODP>::V sh_ws[kPrepWords];
  const int b = blockIdx.x;
  const QuadDesc& d = descs[b];
  const int c = d.c, m = d.m, nact = d.nact;
  const unsigned int p = d.p;
  const size_t tab = (size_t)c * MPAD;
  const unsigned long long N4 = (unsigned long long)c * c * c * c;
  T* tabs = reinterpret_cast<T*>(smem_raw);  // t0 | t1 | t2 | t3, [l][MPAD] each
  unsigned char* cnt = smem_raw + 4 * tab * sizeof(T);
  long long* coef = reinterpret_cast<long long*>(cnt + (N4 + 15) / 16 * 16);
  unsigned char* zf = reinterpret_cast<unsigned char*>(coef + c);
  const long long* __restrict__ tm = stage + d.in_off;
  const long long* __restrict__ gcoef = tm + 4 * (size_t)m;
  {
    DevField<true> RB;
    RB.p = p; RB.m64 = d.m64;
    const unsigned utab = (unsigned)tab;
    for (unsigned e = threadIdx.x; e < 4 * utab; e += kSmallThreads) {
      const unsigned t = e / utab, rem = e - t * utab;
      const unsigned l = rem / MPAD, j = rem - l * MPAD;
      T val = 0;
      if ((int)t < nact && (int)j < m) {
        if (MODP) val = (T)RB.mul((unsigned long long)gcoef[l], (unsigned long long)tm[t * m + j]);
        else val = (T)(gcoef[l] * tm[t * m + j]);
      }
      tabs[e] = val;
    }
  }
  for (int e = threadIdx.x; e < c; e += kSmallThreads) coef[e] = gcoef[e];
  for (int e = threadIdx.x; e < 4 * c; e += kSmallThreads) zf[e] = (e / c < nact) && (gcoef[e % c] == 0);
  if (threadIdx.x < 4) sh_res[threadIdx.x] = threadIdx.x == 0 ? d.seed_key : pack_key(-1, -1, kIdxMask);
  if (threadIdx.x == 0) sh_stop = 0;
  __syncthreads();

  {  // zero counts of every candidate
    const T* t0 = tabs; const T* t1 = t0 + tab; const T* t2 = t1 + tab; const T* t3 = t2 + tab;
    const unsigned nprefix = (unsigned)c * c * c;
    const bool small_p = MODP && p <= 0x80000000u;
    for (unsigned q = threadIdx.x; q < nprefix; q += kSmallThreads) {
      int i, j, k;
      decode_prefix(q, c, i, j, k);
      T nb[MPAD];
#pragma unroll
      for (int e = 0; e < MPAD; ++e) {
        const T a0 = t0[(size_t)i * MPAD + e], a1 = t1[(size_t)j * MPAD + e], a2 = t2[(size_t)k * MPAD + e];
        if (small_p) {  // p <= 2^31: the sum of two residues fits 32 bits -- a third of the instructions of the 64-bit form
          unsigned t32 = (unsigned)a0 + (unsigned)a1;
          t32 -= t32 >= p ? p : 0u;
          t32 += (unsigned)a2;
          t32 -= t32 >= p ? p : 0u;
          nb[e] = (T)(t32 ? p - t32 : 0u);
        } else {
          nb[e] = neg_prefix_sum<T, MODP>(a0, a1, a2, p);
        }
        if (e >= m) nb[e] = pad_sentinel<T, MODP>();
      }
      unsigned char* out = cnt + (size_t)q * c;
      for (int l = 0; l < c; ++l) out[l] = (unsigned char)zero_count(t3 + (size_t)l * MPAD, nb);
    }
  }
  __syncthreads();

  const unsigned nchunks = (unsigned)((N4 + 15) / 16);
  for (int num = 0; num < d.npick; ++num) {
    if (threadIdx.x < 32) {
      const int rc = quad_prepare<MODP>(d, coef, sh_res, num, sh_phi, &sh_nphi, sh_ws);
      if (threadIdx.x == 0) { sh_stop = rc; sh_best = sh_res[num]; }
    }
    __syncthreads();
    if (sh_stop) break;
    const int nphi = sh_nphi;
    const unsigned long long seed = sh_res[num];
    unsigned long long best = seed;
    // A thread owns ~c^4/512 candidates: too few for a running best to filter anything.  Instead it walks ITS candidates in
    // decreasing key order -- the largest key below `limit`, then the filter for that one candidate only -- until one passes.
    // sh_best carries the best admissible key anyone has found so far: a thread stops as soon as its remaining keys fall below it.
    unsigned long long limit = ~0ull;
    for (;;) {
      const unsigned long long floor_key = *reinterpret_cast<volatile unsigned long long*>(&sh_best);
      unsigned long long loc = floor_key;
      int loc_rl1 = (int)(loc >> 48), wi = 0, wj = 0, wk = 0, wl = 0;
      for (unsigned g = threadIdx.x; g < nchunks; g += kSmallThreads) {
        unsigned idx = g * 16u;
        int i, j, k, l;
        decode_index(idx, c, i, j, k, l);
#pragma unroll 1
        for (int e = 0; e < 16; ++e, ++idx) {
          const int rl = (int)cnt[idx];
          if (idx < N4 && rl + 1 >= loc_rl1) {
            const int cl = d.cl_const + zf[i] + zf[c + j] + zf[2 * c + k] + zf[3 * c + l];
            const unsigned long long key = pack_key(rl, cl, kIdxMask - 1ull - idx);
            if (key > loc && key < limit) { loc = key; loc_rl1 = rl + 1; wi = i; wj = j; wk = k; wl = l; }
          }
          if (++l == c) { l = 0; if (++k == c) { k = 0; if (++j == c) { j = 0; ++i; } } }
        }
      }
      if (loc == floor_key) break;  // nothing left in this thread that beats the best known key
      if (independent<MODP>(sh_phi, nphi, coef, p, d.m64, wi, wj, wk, wl)) { best = loc; atomicMax(&sh_best, loc); break; }
      limit = loc;
    }
    block_max<kSmallThreads>(best, threadIdx.x, red, [&](unsigned long long v) { sh_res[num] = v; });  // v >= seed: the seed stays when nothing beats it
    __syncthreads();
  }
  if (threadIdx.x < 4) results[b * 4 + threadIdx.x] = sh_res[threadIdx.x];
  if (threadIdx.x == 0) status[b] = sh_stop == 3 ? 3 : 0;
}

// ---- per-device context: pinned staging, device buffers, a private stream --------------------------------------------------------
struct QuadCtx {
  cudaStream_t st = nullptr;
  unsigned char* h_stage = nullptr; size_t h_cap = 0;  // pinned
  unsigned char* d_stage = nullptr; size_t d_cap = 0;
  unsigned char* d_tables = nullptr; size_t tab_cap = 0;
  unsigned char* d_counts = nullptr; size_t cnt_cap = 0;
  unsigned long long* h_res = nullptr; size_t res_cap = 0;  // pinned: [nprob][4] keys then [nprob] status ints
};
static QuadCtx g_quad[64];

static void quad_release_device(int dev) {
  QuadCtx& q = g_quad[dev];
  if (q.h_stage) cudaFreeHost(q.h_stage);
  if (q.h_res) cudaFreeHost(q.h_res);
  if (q.d_stage) cudaFree(q.d_stage);
  if (q.d_tables) cudaFree(q.d_tables);
  if (q.d_counts) cudaFree(q.d_counts);
  if (q.st) cudaStreamDestroy(q.st);
  q = QuadCtx();
}
void quad_release_all() {
  int prev = 0, n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return; }
  cudaGetDevice(&prev);
  for (int dv = 0; dv < n && dv < 64; ++dv)
    if (g_quad[dv].st || g_quad[dv].d_stage) { cudaSetDevice(dv); cudaDeviceSynchronize(); quad_release_device(dv); }
  cudaSetDevice(prev);
}

template <class P>
static cudaError_t grow_device(P** ptr, size_t* cap, size_t need) {
  if (need <= *cap) return cudaSuccess;
  if (*ptr) { cudaDeviceSynchronize(); cudaFree(*ptr); *ptr = nullptr; *cap = 0; }
  size_t want = need < (1u << 20) ? (1u << 20) : need + need / 4;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(ptr), want);
  if (e != cudaSuccess) { cudaGetLastError(); plo_release_workspace(); want = need; e = cudaMalloc(reinterpret_cast<void**>(ptr), want); }
  if (e == cudaSuccess) *cap = want;
  return e;
}
template <class P>
static cudaError_t grow_pinned(P** ptr, size_t* cap, size_t need) {
  if (need <= *cap) return cudaSuccess;
  if (*ptr) { cudaDeviceSynchronize(); cudaFreeHost(*ptr); *ptr = nullptr; *cap = 0; }
  const size_t want = need < (64u << 10) ? (64u << 10) : need + need / 4;
  cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(ptr), want, cudaHostAllocDefault);
  if (e == cudaSuccess) *cap = want;
  return e;
}

}  // namespace plo

using namespace plo;

extern "C" {

int plo_lincomb_quad(uint32_t p, int m, int nproblems, plo_quad_problem* pr) {
  if (!pr || nproblems < 1 || m < 1) { set_error("plo_lincomb_quad: bad argument"); return PLO_E_ARG; }
  if (m > 64) { set_error("plo_lincomb_quad: m = %d > 64 (use plo_lincomb_search per row)", m); return PLO_E_SHAPE; }
  int rc = check_device();
  if (rc) return rc;
  const int mpad = pad_m(m);
  int dev = 0;
  PLO_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) { set_error("plo_lincomb_quad: device index out of range"); return PLO_E_ARG; }
  QuadCtx& Q = g_quad[dev];
  const int sms = sm_count();

  // ---- pass 1: validate, canonical copies, functionals, widths, sizes -----------------------------------------------------
  struct Prep { std::vector<int64_t> tm, cf; std::vector<long long> phi; int nphi = 0; bool none = false, range = false; int nact = 0, npick = 0; long long cmax = 0; bool has_init = false; int seed_mode = 0; long long seedvec[4] = {0, 0, 0, 0}; };
  std::vector<Prep> prep((size_t)nproblems);
  int width = 4, cmaxall = 0, cminall = 1 << 30;
  size_t inv_words = 0;
  size_t stage_i64 = 0, tab_elems = 0, cnt_bytes = 0, zf_bytes = 0;
  try {
    for (int b = 0; b < nproblems; ++b) {
      plo_quad_problem& q = pr[b];
      if (!q.TM || !q.coeffs || q.n < 1 || q.c < 1 || q.c > 511 || q.off < 0 || q.off >= q.n || (q.off & 3) || q.nprev < 0 || q.nprev > q.n ||
          (q.nprev > 0 && !q.prev_rows) || q.n > 4000) {
        set_error("plo_lincomb_quad: bad argument in problem %d", b);
        return PLO_E_ARG;
      }
      Prep& P = prep[b];
      const int n = q.n, c = q.c, off = q.off;
      P.nact = (n - off) < 4 ? (n - off) : 4;
      P.npick = P.nact - (q.nprev > off ? q.nprev - off : 0);
      if (P.npick < 0) P.npick = 0;
      auto canon = [&](int64_t v) { return canonical(p, v); };
      P.tm.assign((size_t)4 * m, 0);
      for (int t = 0; t < P.nact; ++t) for (int j = 0; j < m; ++j) P.tm[(size_t)t * m + j] = canon(q.TM[(size_t)(off + t) * m + j]);
      P.cf.resize(c);
      for (int l = 0; l < c; ++l) P.cf[l] = canon(q.coeffs[l]);
      std::vector<int64_t> pv((size_t)q.nprev * n);
      for (size_t i = 0; i < pv.size(); ++i) pv[i] = canon(q.prev_rows[i]);
      bool ok;
      if (p) { plo::host::ZpField f((int64_t)p); ok = annihilators(f, n, q.nprev, pv.data(), off, P.nact, P.phi, P.nphi); }
      else { plo::host::QField f; ok = annihilators(f, n, q.nprev, pv.data(), off, P.nact, P.phi, P.nphi); }
      if (!ok) { P.none = true; P.nphi = 0; P.phi.assign(16, 0); }
      P.has_init = !(q.init_rl == -1 && q.init_cl == -1);
      if (q.seed_vec && P.has_init && q.nprev == 0) {  // the device can continue with the seed vector iff it lives on the live positions
        bool live = true;
        for (int i = 0; i < n; ++i) if ((i < off || i >= off + P.nact) && canon(q.seed_vec[i]) != 0) live = false;
        if (live) { P.seed_mode = 1; for (int t = 0; t < P.nact; ++t) P.seedvec[t] = canon(q.seed_vec[off + t]); }
      }
      if (!p) {  // magnitude guards of the exact path
        const unsigned __int128 mc = std::max(max_abs(P.cf.begin(), P.cf.end()), max_abs(P.seedvec, P.seedvec + 4));
        const int w = exact_width(mc, max_abs(P.tm.begin(), P.tm.end()));
        if (!w) { set_error("lincomb quad: integer magnitude bound exceeded"); return PLO_E_RANGE; }
        width = std::max(width, w);
        // images u = Psi.w stay below 2^30: the 3x3 minors of quad_prepare then fit 128 bits with room to spare.  Larger functionals
        // of the previous rows are this problem's alone: it picks no row here and reports PLO_QUAD_RANGE, the caller goes on with
        // plo_lincomb_search (its guard allows |phi| . |coef| . 4 < 2^63); the other problems of the call are not affected.
        if (max_abs(P.phi.begin(), P.phi.end()) * mc * 4 >= ((unsigned __int128)1 << 30)) { P.range = true; P.npick = 0; }
        P.cmax = (long long)mc;
      }
      if (c > cmaxall) cmaxall = c;
      if (c < cminall) cminall = c;
      inv_words += (InvTables::words(mpad, 1 << inv_hash_bits(c), c) + 3) / 4 * 4;
      stage_i64 += (size_t)4 * m + c;
      tab_elems += (size_t)4 * c * mpad;
      cnt_bytes += ((size_t)c * c * c * c + 15) / 16 * 16 + ((size_t)c * c * c + 15) / 16 * 16;
      zf_bytes += ((size_t)4 * c + 15) / 16 * 16;
    }
  } catch (const plo::host::RangeError& e) {
    set_error("lincomb quad: %s", e.what());
    return PLO_E_RANGE;
  }
  if (cnt_bytes > PLO_QUAD_MAX_COUNT_BYTES) { set_error("lincomb quad: %zu bytes of zero counts exceed the limit (use plo_lincomb_search per row)", cnt_bytes); return PLO_E_SHAPE; }

  // ---- layout of the staging buffer: descs | int64 inputs ; device-only tail: zflags | results | status ------------------------
  const size_t desc_bytes = ((size_t)nproblems * sizeof(QuadDesc) + 15) / 16 * 16;
  const size_t in_bytes = (stage_i64 * 8 + 15) / 16 * 16;
  // one block per problem when the tables and counts of the largest fit shared memory; else tables, count and pick kernels, the count
  // by inverse lookup when every problem has many coefficients
  const size_t small_smem = quad_small_smem(cmaxall, mpad, width);
  const bool small = small_smem <= kSmemLimit && getenv("PLO_QUAD_NOSMALL") == nullptr;
  bool use_inv = !small && inv_lookup_applies(p, width, cminall);
  const size_t inv_bytes = use_inv ? inv_words * 4 : 0;
  const size_t h2d_bytes = desc_bytes + in_bytes + inv_bytes;
  const size_t zf_off0 = h2d_bytes;
  const size_t res_off = zf_off0 + zf_bytes;
  const size_t status_off = res_off + (size_t)nproblems * 4 * 8;
  const size_t rhist_off = status_off + ((size_t)nproblems * 4 + 15) / 16 * 16;  // [nproblems][256] histogram of the row maxima (inverse-lookup path)
  const size_t stage_total = rhist_off + (size_t)nproblems * 256 * 4;
  const size_t res_bytes = (size_t)nproblems * 4 * 8 + (size_t)nproblems * 4;
  if (!Q.st) PLO_CUDA(cudaStreamCreateWithFlags(&Q.st, cudaStreamNonBlocking));
  cudaError_t e = grow_pinned(&Q.h_stage, &Q.h_cap, h2d_bytes);
  if (e == cudaSuccess) e = grow_pinned(&Q.h_res, &Q.res_cap, res_bytes);
  if (e == cudaSuccess) e = grow_device(&Q.d_stage, &Q.d_cap, stage_total);
  if (e == cudaSuccess && !small) e = grow_device(&Q.d_tables, &Q.tab_cap, tab_elems * (size_t)width);
  if (e == cudaSuccess && !small) e = grow_device(&Q.d_counts, &Q.cnt_cap, cnt_bytes);
  if (e != cudaSuccess) { set_error("lincomb quad: allocation failed: %s", cudaGetErrorString(e)); cudaGetLastError(); return PLO_E_CUDA; }

  QuadDesc* hd = reinterpret_cast<QuadDesc*>(Q.h_stage);
  long long* hin = reinterpret_cast<long long*>(Q.h_stage + desc_bytes);
  size_t in_off = 0, tab_off = 0, cnt_off = 0, zf_off = 0, inv_off = 0, inv_smem = 0;
  const int max_rows = t3_tile_rows(mpad, width);
  unsigned long long max_items = 1, max_chunks = 1, max_tab = 1;
  for (int b = 0; b < nproblems; ++b) {
    const plo_quad_problem& q = pr[b];
    const Prep& P = prep[b];
    QuadDesc& d = hd[b];
    memset(&d, 0, sizeof(d));
    d.n = q.n; d.m = m; d.c = q.c; d.nact = P.nact; d.mpad = mpad;
    d.cl_const = q.n - P.nact;
    d.nphi0 = P.nphi; d.seed_mode = P.seed_mode; d.p = p; d.npick = P.npick;
    d.tab_off = tab_off; d.cnt_off = cnt_off; d.in_off = in_off; d.zf_off = zf_off;
    d.seed_key = pack_key(q.init_rl, q.init_cl, kIdxMask);
    d.cmax = P.cmax;
    d.m64 = p ? ~0ull / p : 0;
    if (use_inv) {
      d.hbits = inv_hash_bits(q.c);
      d.inv_off = inv_off;
      uint32_t* dst = reinterpret_cast<uint32_t*>(Q.h_stage + desc_bytes + in_bytes) + inv_off;
      if (!build_inv_tables(p, m, mpad, q.c, d.hbits, P.nact == 4 ? P.tm.data() + (size_t)3 * m : nullptr, P.cf.data(), dst)) use_inv = false;
      inv_off += (InvTables::words(mpad, 1 << d.hbits, q.c) + 3) / 4 * 4;
      inv_smem = std::max(inv_smem, inv_smem_bytes(mpad, q.c));
    }
    for (int t = 0; t < 16; ++t) d.phi0[t] = P.phi[t];
    for (int t = 0; t < 4; ++t) d.seedvec[t] = P.seedvec[t];
    // every SM busy even for small c: split the l range of a prefix across threads
    const unsigned long long nprefix = (unsigned long long)q.c * q.c * q.c;
    const int lsplit = lsplit_for(q.c, nproblems, sms);
    d.lsplit = lsplit;
    memcpy(hin + in_off, P.tm.data(), (size_t)4 * m * 8);
    memcpy(hin + in_off + (size_t)4 * m, P.cf.data(), (size_t)q.c * 8);
    in_off += (size_t)4 * m + q.c;
    tab_off += (size_t)4 * q.c * mpad;
    cnt_off += ((size_t)q.c * q.c * q.c * q.c + 15) / 16 * 16 + ((size_t)q.c * q.c * q.c + 15) / 16 * 16;
    zf_off += ((size_t)4 * q.c + 15) / 16 * 16;
    max_items = std::max(max_items, nprefix * lsplit);
    max_chunks = std::max(max_chunks, (nprefix * q.c + 15) / 16);
    max_tab = std::max<unsigned long long>(max_tab, (unsigned long long)4 * q.c * mpad);
  }

  cudaStream_t st = Q.st;
  const bool timing = getenv("PLO_TIMING") != nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  if (timing) { for (auto& x : ev) cudaEventCreate(&x); cudaEventRecord(ev[0], st); }
  PLO_CUDA(cudaMemcpyAsync(Q.d_stage, Q.h_stage, h2d_bytes, cudaMemcpyHostToDevice, st));
  if (timing) cudaEventRecord(ev[1], st);
  const QuadDesc* dd = reinterpret_cast<const QuadDesc*>(Q.d_stage);
  const long long* dstage = reinterpret_cast<const long long*>(Q.d_stage + desc_bytes);
  unsigned char* dzf = Q.d_stage + zf_off0;
  unsigned long long* dres = reinterpret_cast<unsigned long long*>(Q.d_stage + res_off);
  int* dstatus = reinterpret_cast<int*>(Q.d_stage + status_off);
  if (small) {
    e = with_elem(p, width, [&](auto w, auto modp) {
      return with_mpad(mpad, [&](auto mp) {
        return launch(quad_small_kernel<elem_t<decltype(w)::value>, decltype(mp)::value, decltype(modp)::value>, dim3(nproblems), kSmallThreads,
                      small_smem, st, dd, dstage, dres, dstatus);
      });
    });
    if (e != cudaSuccess) { set_error("lincomb quad (one-launch path): %s", cudaGetErrorString(e)); return PLO_E_CUDA; }
  } else {
    // the inverse-lookup tables follow the inputs in the staging buffer; T0..T2 are built times -A3_e^-1 for the lookup
    const bool inv = use_inv && inv_smem <= kSmemLimit;
    const unsigned int* dinv = inv ? reinterpret_cast<const unsigned int*>(Q.d_stage + desc_bytes + in_bytes) : nullptr;
    unsigned int* drhist = inv ? reinterpret_cast<unsigned int*>(Q.d_stage + rhist_off) : nullptr;  // histogram of the row maxima
    e = with_elem(p, width, [&](auto w, auto modp) -> cudaError_t {
      typedef elem_t<decltype(w)::value> T;
      constexpr bool MODP = decltype(modp)::value;
      const dim3 tg((unsigned)std::min<unsigned long long>((max_tab + 255) / 256, 64), nproblems);
      quad_tables_kernel<T, MODP><<<tg, 256, 0, st>>>(dd, dstage, (T*)Q.d_tables, dzf, dres, dstatus, dinv);
      if (inv) {
        const unsigned long long pb = ((unsigned long long)cmaxall * cmaxall * cmaxall + kLcThreads - 1) / kLcThreads;
        const dim3 ig((unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>(pb, (unsigned long long)sms * 8ull)), nproblems);
        const cudaError_t r = cudaMemsetAsync(drhist, 0, (size_t)nproblems * 256 * 4, st);
        if (r != cudaSuccess) return r;
        return with_mpad(mpad, [&](auto mp) {
          return launch(quad_count_inv_kernel<decltype(mp)::value>, ig, kLcThreads, inv_smem, st, dd, (const uint32_t*)Q.d_tables, dinv, Q.d_counts, drhist);
        });
      }
      const int ltile = cmaxall < max_rows ? cmaxall : max_rows;
      const unsigned long long blocks = (max_items + kLcThreads - 1) / kLcThreads;
      const dim3 cg((unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>(blocks, (unsigned long long)sms * 8ull)), nproblems);
      return with_mpad(mpad, [&](auto mp) {
        return launch(quad_count_kernel<T, decltype(mp)::value, MODP>, cg, kLcThreads, (size_t)ltile * mpad * width, st, dd, (const T*)Q.d_tables, Q.d_counts, max_rows);
      });
    });
    if (e != cudaSuccess) { set_error("lincomb quad count launch: %s", cudaGetErrorString(e)); return PLO_E_CUDA; }
    const unsigned long long blocks = (max_chunks + kPickThreads - 1) / kPickThreads;
    const dim3 pg((unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>(blocks, (unsigned long long)sms * 4ull)), nproblems);
    const dim3 pa(std::min<unsigned>(pg.x, (unsigned)sms), nproblems);
    auto pick = p ? quad_pick_kernel<true> : quad_pick_kernel<false>;
    for (int num = 0; num < 4; ++num) {
      // with the histogram: the best rows first (one wave of blocks), then the whole pick, which returns at once when the first found its winner
      if (drhist) pick<<<pa, kPickThreads, 0, st>>>(dd, dstage, dzf, Q.d_counts, dres, dstatus, num, drhist, 1);
      pick<<<pg, kPickThreads, 0, st>>>(dd, dstage, dzf, Q.d_counts, dres, dstatus, num, drhist, drhist ? 2 : 0);
    }
    PLO_CUDA(cudaGetLastError());
  }
  if (timing) cudaEventRecord(ev[2], st);
  PLO_CUDA(cudaMemcpyAsync(Q.h_res, dres, res_bytes, cudaMemcpyDeviceToHost, st));  // keys and status words are contiguous
  if (timing) cudaEventRecord(ev[3], st);
  PLO_CUDA(cudaStreamSynchronize(st));
  if (timing) {
    float a = 0, b2 = 0, c2 = 0;
    cudaEventElapsedTime(&a, ev[0], ev[1]); cudaEventElapsedTime(&b2, ev[1], ev[2]); cudaEventElapsedTime(&c2, ev[2], ev[3]);
    fprintf(stderr, "# [B200] plo_lincomb_quad: %d problems, c <= %d, %s path: h2d %.1f us (%zu B), kernels %.1f us, d2h %.1f us\n", nproblems, cmaxall,
            small ? "one-launch" : "multi-kernel", a * 1e3, h2d_bytes, b2 * 1e3, c2 * 1e3);
    for (auto& x : ev) cudaEventDestroy(x);
  }

  const int* hstatus = reinterpret_cast<const int*>(Q.h_res + (size_t)nproblems * 4);
  for (int b = 0; b < nproblems; ++b) {
    plo_quad_problem& q = pr[b];
    const Prep& P = prep[b];
    q.nrows = 0; q.status = PLO_QUAD_DONE;
    for (int t = 0; t < 4; ++t) { q.rl[t] = -1; q.cl[t] = -1; q.index[t] = PLO_NO_INDEX; }
    if (P.range) { q.status = PLO_QUAD_RANGE; continue; }  // functionals of prev_rows beyond the device filter's guard
    for (int num = 0; num < P.npick; ++num) {
      const unsigned long long key = Q.h_res[(size_t)b * 4 + num];
      const unsigned long long seed = num == 0 ? pack_key(q.init_rl, q.init_cl, kIdxMask) : pack_key(-1, -1, kIdxMask);
      if (key != seed && !P.none) {
        unpack_key(key, q.rl[num], q.cl[num], q.index[num]);
        q.nrows = num + 1;
        continue;
      }
      if (num == 0 && P.has_init) {  // the seed vector keeps row 0 (found starts true, :290-295)
        q.rl[0] = q.init_rl; q.cl[0] = q.init_cl; q.index[0] = PLO_NO_INDEX;
        q.nrows = 1;
        if (!P.seed_mode) { if (P.npick > 1) q.status = PLO_QUAD_SEED; break; }
        continue;
      }
      q.status = hstatus[b] == 3 ? PLO_QUAD_RANGE : PLO_QUAD_MISS;
      break;
    }
  }
  return PLO_OK;
}

}  // extern "C"
