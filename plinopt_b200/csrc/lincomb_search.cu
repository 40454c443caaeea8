// lincomb_search.cu -- sparsifier candidate scoring on sm_100a.
//
// Replaces one (block,num) step of the reference's quad loop
//   include/plinopt_sparsify.inl:299-314  (i,j,k,l over Coeffs^4, l fastest)
// and its per-candidate body testLinComb
//   include/plinopt_sparsify.inl:166-197  (setRow + rank, v = TM^T.w, two
//                                          zero counts, strict '>' keep-best).
//
// Formulation (exact, no multiplications on the device):
//   v(i,j,k,l) = C_i.TM[off] + C_j.TM[off+1] + C_k.TM[off+2] + C_l.TM[off+3]
// The host tabulates the c x m products C_x.TM[off+t] once (4 tables, in the
// field: integers, or residues mod p).  A thread owns a prefix (i,j,k), sums
// three table rows into nb_j = -(base_j) (m registers) and then, for every l,
// counts the coordinates with  T3[l][j] == nb_j  -- one compare per output
// coordinate per candidate, T3 being read warp-uniformly from shared memory.
// The independence filter (rank(Cand) > num) is evaluated lazily, only for a
// candidate that would beat the thread's running best: w is independent of the
// previous rows iff some annihilator functional phi_q of their span has
// phi_q.w != 0 (<= 4 functionals restricted to the 4 live positions).
// Winner = maximum of the packed key (rl, cl, -index): equals the reference's
// strict-'>' first-maximiser rule and is associative, so the warp-shuffle /
// block / atomicMax reduction is deterministic for any launch geometry.
#include <algorithm>
#include <vector>

#include "lincomb_common.cuh"

namespace plo {

template <typename T>
struct LcParams {
  int c, m, lsplit, ltile;
  int rl_const;                 // zero coordinates shared by every candidate (columns of TM that vanish on the live rows; wide path)
  unsigned long long qlo, qhi;  // prefix range (i*c+j)*c+k of this launch (multi-GPU sharding of one search)
  unsigned int p;
  int cl_const;
  unsigned long long m64;       // floor((2^64 - 1) / p): Barrett reductions of the independence test
  const T* t0;   // [b][l][MPAD]
  const T* t1;   // [b][l][MPAD]
  const T* t2;   // [b][MPAD][c]   (transposed: consecutive k coalesce)
  const T* t3;   // [b][l][MPAD]
  const unsigned char* zflag;       // [b][4][c]   coefficient is zero at an active position
  const long long* phi;             // [b][4][4]   annihilator functionals on the live positions
  const int* nphi;                  // [b]
  const long long* coef;            // [b][c]      coefficient values (ints / canonical residues)
  const unsigned long long* seed;   // [b]
  unsigned long long* result;       // [b]
};

template <typename T, int MPAD, bool MODP>
__global__ void __launch_bounds__(kLcThreads) lincomb_kernel(const LcParams<T> prm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* t3s = reinterpret_cast<T*>(smem_raw);
  __shared__ unsigned long long red[32];
  constexpr int VEC = 16 / sizeof(T);  // elements per 128-bit shared load
  const int b = blockIdx.y;
  const int c = prm.c;
  const size_t tab = (size_t)c * MPAD;
  const T* __restrict__ t0 = prm.t0 + b * tab;
  const T* __restrict__ t1 = prm.t1 + b * tab;
  const T* __restrict__ t2 = prm.t2 + b * tab;
  const T* __restrict__ t3 = prm.t3 + b * tab;
  const unsigned char* __restrict__ zf = prm.zflag + (size_t)b * 4 * c;
  const long long* __restrict__ phi = prm.phi + b * 16;
  const long long* __restrict__ coef = prm.coef + (size_t)b * c;
  const int nphi = prm.nphi[b];

  unsigned long long best = prm.seed[b];
  const unsigned long long item0 = prm.qlo * (unsigned long long)prm.lsplit;
  const unsigned long long nitems = prm.qhi * (unsigned long long)prm.lsplit;
  const unsigned long long nthreads = (unsigned long long)gridDim.x * kLcThreads;

  for (int l0 = 0; l0 < c; l0 += prm.ltile) {
    const int l1 = min(c, l0 + prm.ltile);
    __syncthreads();
    {  // stage the T3 tile
      const uint4* src = reinterpret_cast<const uint4*>(t3 + (size_t)l0 * MPAD);
      uint4* dst = reinterpret_cast<uint4*>(t3s);
      const int nvec = (l1 - l0) * MPAD / VEC;
      for (int e = threadIdx.x; e < nvec; e += kLcThreads) dst[e] = src[e];
    }
    __syncthreads();
    const int lc = (l1 - l0 + prm.lsplit - 1) / prm.lsplit;
    for (unsigned long long item = item0 + (unsigned long long)blockIdx.x * kLcThreads + threadIdx.x; item < nitems; item += nthreads) {
      const unsigned long long q = item / (unsigned)prm.lsplit;
      const int s = (int)(item - q * (unsigned)prm.lsplit);
      const int la = l0 + s * lc, lb = min(l1, la + lc);
      if (la >= lb) continue;
      int i, j, k;
      decode_prefix(q, c, i, j, k);
      T nb[MPAD];
#pragma unroll
      for (int e = 0; e < MPAD; ++e) {
        const T a0 = t0[(size_t)i * MPAD + e], a1 = t1[(size_t)j * MPAD + e], a2 = t2[(size_t)e * c + k];
        nb[e] = neg_prefix_sum<T, MODP>(a0, a1, a2, prm.p);
        if (e >= prm.m) nb[e] = pad_sentinel<T, MODP>();
      }
      const int zc = prm.cl_const + zf[i] + zf[c + j] + zf[2 * c + k];
      int best_rl1 = (int)(best >> 48);  // rl+1 of the running best
      for (int l = la; l < lb; ++l) {
        const int rl = zero_count(t3s + (size_t)(l - l0) * MPAD, nb);
        if (rl + 1 >= best_rl1) {
          const int cl = zc + zf[3 * c + l];
          const unsigned long long idx = q * (unsigned)c + (unsigned)l;
          const unsigned long long key = pack_key(rl, cl, kIdxMask - 1ull - idx);
          if (key > best && independent<MODP>(phi, nphi, coef, prm.p, prm.m64, i, j, k, l)) {
            best = key;
            best_rl1 = rl + 1;
          }
        }
      }
    }
  }
  block_max<kLcThreads>(best, threadIdx.x, red, [&](unsigned long long v) { atomicMax(prm.result + b, v); });  // one atomicMax per block
}

// ---------------------------------------------------------------------------
// Many coefficients mod p (c >= 32): inverse lookup instead of c compares per coordinate (lincomb_common.cuh, "inverse lookup").
// Thread <-> prefix; per coordinate one Barrett multiplication and one hash probe; the hits go into c byte counters of the
// thread (shared memory, padded rows); then the usual keep-best over l, skipping four empty counters at a time.
// Same key, same lazy independence test, same winner as lincomb_kernel.
// ---------------------------------------------------------------------------
struct LcInvParams {
  const unsigned int* inv;   // [b][InvTables::words]
  int hbits, cpad;           // hash bits; c rounded up to a multiple of 4
};

template <int MPAD>
__global__ void __launch_bounds__(kLcThreads) lincomb_inv_kernel(const LcParams<unsigned int> prm, const LcInvParams ip) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned long long red[32];
  const int b = blockIdx.y, c = prm.c, hsize = 1 << ip.hbits;
  const unsigned int p = prm.p;
  unsigned int* ninv = reinterpret_cast<unsigned int*>(smem_raw);
  uint2* htab = reinterpret_cast<uint2*>(ninv + MPAD);
  unsigned int* nextdup = reinterpret_cast<unsigned int*>(htab + hsize);
  unsigned char* hist0 = reinterpret_cast<unsigned char*>(nextdup + c);
  const int hstride = ip.cpad + 4;  // bytes per thread: consecutive threads start in different banks
  unsigned char* hist = hist0 + (size_t)threadIdx.x * hstride;
  {
    const unsigned int* src = ip.inv + (size_t)b * InvTables::words(MPAD, hsize, c);
    const int nw = (int)InvTables::words(MPAD, hsize, c);
    for (int e = threadIdx.x; e < nw; e += kLcThreads) ninv[e] = src[e];  // ninv | htab | nextdup are contiguous
  }
  __syncthreads();
  const InvShared sh = inv_shared_addresses(ninv, htab, nextdup, hist);
  const size_t tab = (size_t)c * MPAD;
  const unsigned int* __restrict__ t0 = prm.t0 + b * tab;
  const unsigned int* __restrict__ t1 = prm.t1 + b * tab;
  const unsigned int* __restrict__ t2 = prm.t2 + b * tab;
  const unsigned char* __restrict__ zf = prm.zflag + (size_t)b * 4 * c;
  const long long* __restrict__ phi = prm.phi + b * 16;
  const long long* __restrict__ coef = prm.coef + (size_t)b * c;
  const int nphi = prm.nphi[b];
  unsigned long long best = prm.seed[b];
  const unsigned long long nthreads = (unsigned long long)gridDim.x * kLcThreads;
  for (unsigned long long q = prm.qlo + (unsigned long long)blockIdx.x * kLcThreads + threadIdx.x; q < prm.qhi; q += nthreads) {
    int i, j, k;
    decode_prefix(q, c, i, j, k);
    for (int w = 0; w < ip.cpad; w += 4) *reinterpret_cast<unsigned int*>(hist + w) = 0u;
    // the counting loop is shared with quad_count_inv_kernel (lincomb_common.cuh).  It is NOT fully unrolled: nothing is kept per
    // coordinate, and 48 copies of the probe loop overflow the instruction cache (ncu: stall reason no_instruction 7.7 warps per issue
    // with the unrolled body).  A register list of hits instead of the byte counters was tried and is slower: with Hopcroft-Musinski
    // data hits are common (structured prefixes), not rare.
    const int base = (int)inv_count_prefix(t0 + (size_t)i * MPAD, t1 + (size_t)j * MPAD, t2 + k, c, prm.m, p, ip.hbits, sh);
    const int zc = prm.cl_const + zf[i] + zf[c + j] + zf[2 * c + k];
    int best_rl1 = (int)(best >> 48);
    for (int l0 = 0; l0 < c; l0 += 4) {
      const unsigned int w = *reinterpret_cast<const unsigned int*>(hist + l0);
      if (w == 0u && base + 1 < best_rl1) continue;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int l = l0 + t;
        if (l >= c) break;
        const int rl = base + (int)((w >> (8 * t)) & 0xFFu);
        if (rl + 1 >= best_rl1) {
          const int cl = zc + zf[3 * c + l];
          const unsigned long long idx = q * (unsigned)c + (unsigned)l;
          const unsigned long long key = pack_key(rl, cl, kIdxMask - 1ull - idx);
          if (key > best && independent<true>(phi, nphi, coef, p, prm.m64, i, j, k, l)) {
            best = key;
            best_rl1 = rl + 1;
          }
        }
      }
    }
  }
  block_max<kLcThreads>(best, threadIdx.x, red, [&](unsigned long long v) { atomicMax(prm.result + b, v); });
}

// ---------------------------------------------------------------------------
// Wide outputs (m > 64, e.g. 32x32x32_15096: TM is 4 x 15096).  The m coordinates are cut into tiles of 64;
// a block stages the T3 rows of one tile in shared memory and every thread sweeps prefixes (i,j,k) against it
// exactly as above, but a candidate's zero count is now spread over the tiles: partial counts are accumulated
// with one RED per (candidate, tile) into counts[c^4]; lincomb_big_pick_kernel then applies the keep-best rule.
// ---------------------------------------------------------------------------
constexpr int kBigTile = 64;

template <typename T, bool MODP>
__global__ void __launch_bounds__(kLcThreads) lincomb_big_count_kernel(const LcParams<T> prm, int mpad, int tiles_per_group,
                                                                       unsigned int* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* t3s = reinterpret_cast<T*>(smem_raw);  // [c][64]
  constexpr int VEC = 16 / sizeof(T);
  const int b = blockIdx.z, c = prm.c;
  const size_t tab = (size_t)c * mpad;
  const T* __restrict__ t0 = prm.t0 + b * tab;
  const T* __restrict__ t1 = prm.t1 + b * tab;
  const T* __restrict__ t2 = prm.t2 + b * tab;
  const T* __restrict__ t3 = prm.t3 + b * tab;
  unsigned int* __restrict__ cnt = counts + (size_t)b * c * c * c * c;
  const int ntiles = mpad / kBigTile;
  const int tile0 = blockIdx.y * tiles_per_group, tile1 = min(ntiles, tile0 + tiles_per_group);
  const unsigned long long nthreads = (unsigned long long)gridDim.x * kLcThreads;
  for (int tile = tile0; tile < tile1; ++tile) {
    __syncthreads();
    for (int e = threadIdx.x; e < c * kBigTile / VEC; e += kLcThreads) {
      const int l = e / (kBigTile / VEC), v = e % (kBigTile / VEC);
      reinterpret_cast<uint4*>(t3s)[e] = reinterpret_cast<const uint4*>(t3 + (size_t)l * mpad + (size_t)tile * kBigTile)[v];
    }
    __syncthreads();
    for (unsigned long long q = prm.qlo + (unsigned long long)blockIdx.x * kLcThreads + threadIdx.x; q < prm.qhi; q += nthreads) {
      int i, j, k;
      decode_prefix(q, c, i, j, k);
      T nb[kBigTile];
#pragma unroll
      for (int e = 0; e < kBigTile; ++e) {
        const int col = tile * kBigTile + e;
        const T a0 = t0[(size_t)i * mpad + col], a1 = t1[(size_t)j * mpad + col], a2 = t2[(size_t)col * c + k];
        nb[e] = neg_prefix_sum<T, MODP>(a0, a1, a2, prm.p);
        if (col >= prm.m) nb[e] = pad_sentinel<T, MODP>();
      }
      for (int l = 0; l < c; ++l) {
        const int rl = zero_count(t3s + (size_t)l * kBigTile, nb);
        if (rl) atomicAdd(cnt + q * (unsigned)c + (unsigned)l, (unsigned)rl);
      }
    }
  }
}

template <typename T, bool MODP>
__global__ void __launch_bounds__(kLcThreads) lincomb_big_pick_kernel(const LcParams<T> prm, const unsigned int* __restrict__ counts) {
  __shared__ unsigned long long red[32];
  const int b = blockIdx.y, c = prm.c;
  const unsigned char* __restrict__ zf = prm.zflag + (size_t)b * 4 * c;
  const long long* __restrict__ phi = prm.phi + b * 16;
  const long long* __restrict__ coef = prm.coef + (size_t)b * c;
  const int nphi = prm.nphi[b];
  const unsigned int* __restrict__ cnt = counts + (size_t)b * c * c * c * c;
  unsigned long long best = prm.seed[b];
  const unsigned long long lo = prm.qlo * (unsigned)c, hi = prm.qhi * (unsigned)c;
  for (unsigned long long idx = lo + (unsigned long long)blockIdx.x * kLcThreads + threadIdx.x; idx < hi; idx += (unsigned long long)gridDim.x * kLcThreads) {
    int i, j, k, l;
    decode_index(idx, c, i, j, k, l);
    const int rl = (int)cnt[idx] + prm.rl_const;
    const int cl = prm.cl_const + zf[i] + zf[c + j] + zf[2 * c + k] + zf[3 * c + l];
    const unsigned long long key = pack_key(rl, cl, kIdxMask - 1ull - idx);
    if (key > best && independent<MODP>(phi, nphi, coef, prm.p, prm.m64, i, j, k, l)) best = key;
  }
  block_max<kLcThreads>(best, threadIdx.x, red, [&](unsigned long long v) { atomicMax(prm.result + b, v); });
}

__global__ void lincomb_init_kernel(unsigned long long* result, const unsigned long long* seed, int nbatch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nbatch) result[b] = seed[b];
}

}  // namespace plo

using namespace plo;

struct plo_lincomb_plan {
  uint32_t p;
  int nbatch, n, m, off, c, nprev, mpad, width;  // width: 4 or 8 bytes per element
  std::vector<unsigned long long> h_seed;
  std::vector<int> h_init_rl, h_init_cl;
  std::vector<char> trivially_none;  // previous rows dependent: no admissible candidate
  void* d_tables;                    // t0 | t1 | t2 | t3
  unsigned char* d_zflag;
  long long* d_phi;
  int* d_nphi;
  long long* d_coef;
  unsigned long long *d_seed, *d_result;
  int lsplit, ltile, grid;
  size_t smem;
  bool big;                // m > 64: tiled count + pick kernels
  unsigned int* d_counts;  // [nbatch][c^4] zero counts (big path)
  int tiles_per_group, tile_groups;
  int m_eff, rl_const;     // wide path: columns kept after dropping those that vanish on the live rows
  bool use_inv;            // mod p, c >= 32: inverse-lookup kernel
  unsigned int* d_inv;
  int hbits;
  size_t inv_smem;
};

namespace {

template <typename T>
void fill_tables(uint32_t p, int n, int m, int off, int nact, int c, int mpad, const int64_t* TM, const int64_t* coef,
                 T* t0, T* t1, T* t2, T* t3) {
  const size_t tab = (size_t)c * mpad;
  T* tabs[4] = {t0, t1, t2, t3};
  for (int t = 0; t < 4; ++t) std::fill(tabs[t], tabs[t] + tab, (T)0);
  for (int t = 0; t < nact; ++t) {
    const int64_t* row = TM + (size_t)(off + t) * m;
    for (int l = 0; l < c; ++l)
      for (int j = 0; j < m; ++j) {
        T val;
        if (p) val = (T)(((unsigned __int128)(uint64_t)coef[l] * (uint64_t)row[j]) % p);
        else val = (T)(coef[l] * row[j]);
        if (t == 2) t2[(size_t)j * c + l] = val;
        else tabs[t][(size_t)l * mpad + j] = val;
      }
  }
  (void)n;
}

}  // namespace

extern "C" {

void plo_lincomb_plan_destroy(plo_lincomb_plan* pl) {
  if (!pl) return;
  pool_free(pl->d_tables); pool_free(pl->d_zflag); pool_free(pl->d_phi); pool_free(pl->d_nphi);
  pool_free(pl->d_coef); pool_free(pl->d_seed); pool_free(pl->d_result); pool_free(pl->d_counts); pool_free(pl->d_inv);
  delete pl;
}

int plo_lincomb_plan_create(plo_lincomb_plan** plan, uint32_t p, int nbatch, int n, int m, const int64_t* TM, int off,
                            int c, const int64_t* coeffs, int nprev, const int64_t* prev_rows, const int* init_rl,
                            const int* init_cl) {
  if (!plan || !TM || !coeffs || nbatch < 1 || n < 1 || m < 1 || c < 1 || c > 511 || off < 0 || off >= n || (off & 3) ||
      nprev < 0 || nprev > n || (nprev > 0 && !prev_rows) || n > 4000 || m > 65000) {
    set_error("plo_lincomb_plan_create: bad argument");
    return PLO_E_ARG;
  }
  int rc = check_device();
  if (rc) return rc;
  const bool big = m > 64;
  int mpad = big ? (m + kBigTile - 1) / kBigTile * kBigTile : pad_m(m);
  const int nact = (n - off) < 4 ? (n - off) : 4;
  if (big && (c > 64 || (unsigned long long)nbatch * c * c * c * c > (1ull << 28))) {
    set_error("lincomb search: m = %d > 64 needs c <= 64 and nbatch * c^4 <= 2^28", m);
    return PLO_E_SHAPE;
  }

  // canonical copies
  std::vector<int64_t> tm((size_t)nbatch * n * m), cf((size_t)nbatch * c), pv((size_t)nbatch * nprev * n);
  for (size_t i = 0; i < tm.size(); ++i) tm[i] = canonical(p, TM[i]);
  for (size_t i = 0; i < cf.size(); ++i) cf[i] = canonical(p, coeffs[i]);
  for (size_t i = 0; i < pv.size(); ++i) pv[i] = canonical(p, prev_rows[i]);

  // wide path: a column of TM that is zero on the live rows off..off+nact-1 is a zero coordinate of EVERY candidate; such
  // columns are dropped from the tables and counted once (HM matrices are sparse: 70 % of the 15096 columns for C5)
  int m_eff = m, rl_const = 0;
  if (big) {
    std::vector<std::vector<int>> keep(nbatch);
    m_eff = 1;
    for (int b = 0; b < nbatch; ++b) {
      for (int j = 0; j < m; ++j) {
        bool nz = false;
        for (int t = 0; t < nact && !nz; ++t) nz = tm[((size_t)b * n + off + t) * m + j] != 0;
        if (nz) keep[b].push_back(j);
      }
      if ((int)keep[b].size() > m_eff) m_eff = (int)keep[b].size();
    }
    std::vector<int64_t> tmc((size_t)nbatch * n * m_eff, 0);
    for (int b = 0; b < nbatch; ++b)
      for (int t = 0; t < nact; ++t)
        for (size_t q = 0; q < keep[b].size(); ++q) tmc[((size_t)b * n + off + t) * m_eff + q] = tm[((size_t)b * n + off + t) * m + keep[b][q]];
    tm.swap(tmc);
    rl_const = m - m_eff;  // dropped columns, minus the all-zero padding columns of the shorter problems (counted by the kernel)
  }
  const int m_tab = m_eff;  // row length of the tables
  if (big) mpad = (m_eff + kBigTile - 1) / kBigTile * kBigTile;
  int width = 4;
  if (!p) {  // exact integers: magnitude guard over the live rows
    unsigned __int128 mt = 0;
    for (int b = 0; b < nbatch; ++b) {
      const int64_t* live = tm.data() + ((size_t)b * n + off) * m_tab;
      mt = std::max(mt, max_abs(live, live + (size_t)nact * m_tab));
    }
    width = exact_width(max_abs(cf.begin(), cf.end()), mt);
    if (!width) { set_error("lincomb search: integer magnitude bound exceeded"); return PLO_E_RANGE; }
  }

  plo_lincomb_plan* pl = new plo_lincomb_plan();
  pl->p = p; pl->nbatch = nbatch; pl->n = n; pl->m = m; pl->off = off; pl->c = c; pl->nprev = nprev; pl->mpad = mpad; pl->width = width;
  pl->big = big; pl->m_eff = m_eff; pl->rl_const = rl_const; pl->d_counts = nullptr; pl->tiles_per_group = 1; pl->tile_groups = 1;
  pl->use_inv = false; pl->d_inv = nullptr; pl->hbits = 0; pl->inv_smem = 0;
  pl->d_tables = nullptr; pl->d_zflag = nullptr; pl->d_phi = nullptr; pl->d_nphi = nullptr; pl->d_coef = nullptr; pl->d_seed = nullptr; pl->d_result = nullptr;
  pl->h_init_rl.assign(init_rl ? init_rl : nullptr, init_rl ? init_rl + nbatch : nullptr);
  pl->h_init_cl.assign(init_cl ? init_cl : nullptr, init_cl ? init_cl + nbatch : nullptr);
  if (!init_rl) pl->h_init_rl.assign(nbatch, -1);
  if (!init_cl) pl->h_init_cl.assign(nbatch, -1);
  pl->h_seed.resize(nbatch);
  pl->trivially_none.assign(nbatch, 0);

  const size_t tab = (size_t)c * mpad;
  std::vector<unsigned char> tables((size_t)nbatch * 4 * tab * width), zflag((size_t)nbatch * 4 * c, 0);
  std::vector<long long> phi((size_t)nbatch * 16, 0);
  std::vector<int> nphi(nbatch, 0);
  try {
    for (int b = 0; b < nbatch; ++b) {
      const int64_t* tmb = tm.data() + (size_t)b * n * m_tab;
      const int64_t* cfb = cf.data() + (size_t)b * c;
      unsigned char* base = tables.data();
      const size_t per = (size_t)nbatch * tab * width;  // bytes per table kind
      with_elem(p, width, [&](auto w, auto) {
        typedef elem_t<decltype(w)::value> T;
        fill_tables<T>(p, n, m_tab, off, nact, c, mpad, tmb, cfb, (T*)(base + 0 * per) + b * tab, (T*)(base + 1 * per) + b * tab,
                       (T*)(base + 2 * per) + b * tab, (T*)(base + 3 * per) + b * tab);
      });
      for (int t = 0; t < nact; ++t)
        for (int l = 0; l < c; ++l) zflag[((size_t)b * 4 + t) * c + l] = (cfb[l] == 0);
      std::vector<long long> ph;
      int np = 0;
      bool ok;
      if (p) { plo::host::ZpField f((int64_t)p); ok = annihilators(f, n, nprev, pv.data() + (size_t)b * nprev * n, off, nact, ph, np); }
      else { plo::host::QField f; ok = annihilators(f, n, nprev, pv.data() + (size_t)b * nprev * n, off, nact, ph, np); }
      if (!ok) { pl->trivially_none[b] = 1; np = 0; ph.assign(16, 0); }
      if (!p) {  // the device evaluates phi . w in int64: 4 . |phi| . |coef| must stay below 2^63
        if (max_abs(ph.begin(), ph.end()) * max_abs(cfb, cfb + c) * 4 >= ((unsigned __int128)1 << 63)) throw plo::host::RangeError("annihilator functional times coefficient exceeds 63 bits");
      }
      std::copy(ph.begin(), ph.end(), phi.begin() + (size_t)b * 16);
      nphi[b] = np;
      pl->h_seed[b] = pack_key(pl->h_init_rl[b], pl->h_init_cl[b], kIdxMask);
    }
  } catch (const plo::host::RangeError& e) {
    set_error("lincomb search: %s", e.what());
    delete pl;
    return PLO_E_RANGE;
  }

  // launch geometry: all SMs busy even for small c (split the l range across threads)
  const int sms = sm_count();
  const unsigned long long nprefix = (unsigned long long)c * c * c;
  const int lsplit = lsplit_for(c, nbatch, sms);
  pl->lsplit = lsplit;
  const int max_rows = (int)(65536 / ((size_t)mpad * width));
  pl->ltile = c < max_rows ? c : max_rows;
  pl->smem = (size_t)pl->ltile * mpad * width;
  unsigned long long blocks = (nprefix * lsplit + kLcThreads - 1) / kLcThreads;
  const unsigned long long cap = (unsigned long long)sms * 8ull;
  pl->grid = (int)(blocks < cap ? blocks : cap);
  if (pl->grid < 1) pl->grid = 1;

  if (big) {
    const int ntiles = mpad / kBigTile;
    // enough (prefix block, tile group) pairs to fill the machine; a group sweeps its tiles one after the other
    const unsigned long long pblocks = (nprefix + kLcThreads - 1) / kLcThreads;
    int groups = (int)std::min<unsigned long long>((unsigned long long)ntiles, std::max<unsigned long long>(1, (unsigned long long)sms * 4ull / (pblocks * nbatch)));
    pl->tiles_per_group = (ntiles + groups - 1) / groups;
    pl->tile_groups = (ntiles + pl->tiles_per_group - 1) / pl->tiles_per_group;
    pl->grid = (int)std::min<unsigned long long>(pblocks, (unsigned long long)sms * 8ull);
    pl->smem = (size_t)c * kBigTile * width;
    if (pool_alloc(&pl->d_counts, (size_t)nbatch * c * c * c * c * 4) != cudaSuccess) {
      set_error("lincomb search: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
      plo_lincomb_plan_destroy(pl);
      return PLO_E_CUDA;
    }
  }
  auto up = [&](void** dst, const void* src, size_t bytes) -> bool {
    if (pool_alloc(dst, bytes ? bytes : 1) != cudaSuccess) return false;
    return cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  if (!big && inv_lookup_applies(p, width, c)) {
    pl->hbits = inv_hash_bits(c);
    const size_t words = InvTables::words(mpad, 1 << pl->hbits, c);
    std::vector<uint32_t> inv((size_t)nbatch * words);
    bool good = true;
    for (int b = 0; b < nbatch && good; ++b)
      good = build_inv_tables(p, m, mpad, c, pl->hbits, nact == 4 ? tm.data() + ((size_t)b * n + off + 3) * m : nullptr, cf.data() + (size_t)b * c,
                              inv.data() + (size_t)b * words);
    pl->inv_smem = inv_smem_bytes(mpad, c);
    if (good && pl->inv_smem <= kSmemLimit) {
      if (!up((void**)&pl->d_inv, inv.data(), inv.size() * 4)) { set_error("lincomb plan: cudaMalloc failed"); plo_lincomb_plan_destroy(pl); return PLO_E_CUDA; }
      pl->use_inv = true;
      {  // the lookup kernel reads T0, T1, T2 pre-multiplied by -A3_e^-1 (lincomb_common.cuh)
        const size_t per = (size_t)nbatch * tab;  // words per table kind
        uint32_t* base = reinterpret_cast<uint32_t*>(tables.data());
        for (int b = 0; b < nbatch; ++b)
          fold_inv_into_tables((uint32_t)p, m_tab, mpad, c, inv.data() + (size_t)b * words, base + 0 * per + (size_t)b * tab, base + 1 * per + (size_t)b * tab,
                               base + 2 * per + (size_t)b * tab);
      }
      const unsigned long long blocks = (nprefix + kLcThreads - 1) / kLcThreads;
      pl->grid = (int)std::max<unsigned long long>(1, std::min<unsigned long long>(blocks, (unsigned long long)sms * 8ull));
    }
  }
  bool ok = up(&pl->d_tables, tables.data(), tables.size()) && up((void**)&pl->d_zflag, zflag.data(), zflag.size()) &&
            up((void**)&pl->d_phi, phi.data(), phi.size() * 8) && up((void**)&pl->d_nphi, nphi.data(), nphi.size() * 4) &&
            up((void**)&pl->d_coef, cf.data(), cf.size() * 8) && up((void**)&pl->d_seed, pl->h_seed.data(), pl->h_seed.size() * 8) &&
            pool_alloc(&pl->d_result, (size_t)nbatch * 8) == cudaSuccess;
  if (!ok) {
    set_error("lincomb search: device allocation/copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    plo_lincomb_plan_destroy(pl);
    return PLO_E_CUDA;
  }
  *plan = pl;
  return PLO_OK;
}

int plo_lincomb_plan_run(plo_lincomb_plan* pl, void* stream) {
  if (!pl) { set_error("plo_lincomb_plan_run: null plan"); return PLO_E_ARG; }
  return plo_lincomb_plan_run_range(pl, 0, (uint64_t)pl->c * pl->c * pl->c, stream);
}

int plo_lincomb_plan_run_range(plo_lincomb_plan* pl, uint64_t prefix_lo, uint64_t prefix_hi, void* stream) {
  if (!pl) { set_error("plo_lincomb_plan_run_range: null plan"); return PLO_E_ARG; }
  const uint64_t nprefix = (uint64_t)pl->c * pl->c * pl->c;
  if (prefix_hi > nprefix) prefix_hi = nprefix;
  if (prefix_lo > prefix_hi) prefix_lo = prefix_hi;
  cudaStream_t st = (cudaStream_t)stream;
  lincomb_init_kernel<<<(pl->nbatch + 127) / 128, 128, 0, st>>>(pl->d_result, pl->d_seed, pl->nbatch);
  const size_t tab = (size_t)pl->c * pl->mpad;
  const size_t per = (size_t)pl->nbatch * tab;  // elements per table kind
  const dim3 grid(pl->grid, pl->nbatch);
  const cudaError_t e = with_elem(pl->p, pl->width, [&](auto w, auto modp) -> cudaError_t {
    typedef elem_t<decltype(w)::value> T;
    constexpr bool MODP = decltype(modp)::value;
    const T* base = (const T*)pl->d_tables;
    LcParams<T> prm;
    prm.c = pl->c; prm.m = pl->big ? pl->m_eff : pl->m; prm.rl_const = pl->big ? pl->rl_const : 0; prm.lsplit = pl->lsplit; prm.ltile = pl->ltile;
    prm.qlo = prefix_lo; prm.qhi = prefix_hi;
    prm.p = pl->p; prm.cl_const = pl->n - ((pl->n - pl->off) < 4 ? (pl->n - pl->off) : 4); prm.m64 = pl->p ? ~0ull / pl->p : 0;
    prm.t0 = base; prm.t1 = base + per; prm.t2 = base + 2 * per; prm.t3 = base + 3 * per;
    prm.zflag = pl->d_zflag; prm.phi = pl->d_phi; prm.nphi = pl->d_nphi; prm.coef = pl->d_coef;
    prm.seed = pl->d_seed; prm.result = pl->d_result;
    if (pl->big) {
      const size_t c4 = (size_t)pl->c * pl->c * pl->c * pl->c;
      cudaError_t r = cudaMemsetAsync(pl->d_counts, 0, (size_t)pl->nbatch * c4 * 4, st);
      const dim3 cgrid(pl->grid, pl->tile_groups, pl->nbatch);
      const unsigned long long ncand = (prefix_hi - prefix_lo) * (unsigned long long)pl->c;
      const dim3 pgrid((unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>((ncand + kLcThreads - 1) / kLcThreads, (unsigned long long)sm_count() * 8ull)), pl->nbatch);
      if (r == cudaSuccess) r = launch(lincomb_big_count_kernel<T, MODP>, cgrid, kLcThreads, pl->smem, st, prm, pl->mpad, pl->tiles_per_group, pl->d_counts);
      if (r == cudaSuccess) r = launch(lincomb_big_pick_kernel<T, MODP>, pgrid, kLcThreads, 0, st, prm, pl->d_counts);
      return r;
    }
    return with_mpad(pl->mpad, [&](auto mp) {
      constexpr int MPAD = decltype(mp)::value;
      if constexpr (MODP) {
        if (pl->use_inv) {
          LcInvParams ip;
          ip.inv = pl->d_inv; ip.hbits = pl->hbits; ip.cpad = (pl->c + 3) & ~3;
          return launch(lincomb_inv_kernel<MPAD>, grid, kLcThreads, pl->inv_smem, st, prm, ip);
        }
      }
      return launch(lincomb_kernel<T, MPAD, MODP>, grid, kLcThreads, pl->smem, st, prm);
    });
  });
  if (e != cudaSuccess) { set_error("lincomb kernel launch: %s", cudaGetErrorString(e)); return PLO_E_CUDA; }
  return PLO_OK;
}

int plo_lincomb_plan_launches(const plo_lincomb_plan* pl) { return pl && pl->big ? 3 : 2; }

uint64_t plo_lincomb_plan_candidates(const plo_lincomb_plan* pl) {
  return pl ? (uint64_t)pl->nbatch * pl->c * pl->c * pl->c * pl->c : 0;
}

int plo_lincomb_plan_result(plo_lincomb_plan* pl, void* stream, int* best_rl, int* best_cl, uint64_t* best_index) {
  if (!pl || !best_rl || !best_cl || !best_index) { set_error("plo_lincomb_plan_result: bad argument"); return PLO_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<unsigned long long> keys(pl->nbatch);
  PLO_CUDA(cudaMemcpyAsync(keys.data(), pl->d_result, keys.size() * 8, cudaMemcpyDeviceToHost, st));
  PLO_CUDA(cudaStreamSynchronize(st));
  for (int b = 0; b < pl->nbatch; ++b) {
    const unsigned long long key = keys[b];
    if (key == pl->h_seed[b] || pl->trivially_none[b]) {
      best_rl[b] = pl->h_init_rl[b]; best_cl[b] = pl->h_init_cl[b]; best_index[b] = PLO_NO_INDEX;
    } else {
      unpack_key(key, best_rl[b], best_cl[b], best_index[b]);
    }
  }
  return PLO_OK;
}

int plo_lincomb_search_batch(uint32_t p, int nbatch, int n, int m, const int64_t* TM, int off, int c,
                             const int64_t* coeffs, int nprev, const int64_t* prev_rows, const int* init_rl,
                             const int* init_cl, int* best_rl, int* best_cl, uint64_t* best_index) {
  plo_lincomb_plan* pl = nullptr;
  int rc = plo_lincomb_plan_create(&pl, p, nbatch, n, m, TM, off, c, coeffs, nprev, prev_rows, init_rl, init_cl);
  if (rc) return rc;
  rc = plo_lincomb_plan_run(pl, nullptr);
  if (!rc) rc = plo_lincomb_plan_result(pl, nullptr, best_rl, best_cl, best_index);
  plo_lincomb_plan_destroy(pl);
  return rc;
}

int plo_lincomb_search(uint32_t p, int n, int m, const int64_t* TM, int off, int c, const int64_t* coeffs,
                       int nprev, const int64_t* prev_rows, int init_rl, int init_cl,
                       int* best_rl, int* best_cl, uint64_t* best_index) {
  return plo_lincomb_search_batch(p, 1, n, m, TM, off, c, coeffs, nprev, prev_rows, &init_rl, &init_cl, best_rl, best_cl, best_index);
}

}  // extern "C"
