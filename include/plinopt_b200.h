/* =============================================================================
 * plinopt_b200.h -- C ABI of the B200-native candidate-search engine.
 *
 * Drop-in boundary for PLinOpt's one data-parallel hot path (SURVEY.md section 8b).
 * The reference has no FFI; these entry points are what a maintainer binds from
 * the reference's template functions (INTEGRATION.md shows the shims).  Plain
 * pointers and sizes only, caller-owned buffers, int return codes, no
 * exceptions, no torch types.  All reference citations are file:line relative
 * to the reference root.
 *
 * Return codes: 0 success; PLO_E_* (< 0) on argument / CUDA errors (message via
 * plo_last_error()).  Verdict-returning calls document their positive codes.
 *
 * Threading (as in the reference, include/plinopt_sparsify.inl / src/orbiter.cpp: the search entry points are called from ONE host
 * thread, the parallelism is inside): calls are serialised per device by the caller.  The orbit kernels keep L|R|P and the Philox
 * round keys of the plan that ran last in the device's constant memory (re-uploaded when another plan runs), and the workspace
 * pool is per device, so two host threads must not drive the same device at the same time; different devices are independent
 * (plo_orbit_sweep_devices drives several from one thread).  ONE thread may use several streams and alternate plans freely: the bank
 * is guarded by an event (a stream that re-writes it, or reads it after another stream wrote it, waits for its last use).
 * The last-error message is thread-local.
 * ========================================================================== */
#ifndef PLINOPT_B200_H
#define PLINOPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLO_OK 0
#define PLO_E_ARG (-1)      /* bad argument (null pointer, size out of range)            */
#define PLO_E_CUDA (-2)     /* CUDA runtime error, see plo_last_error()                  */
#define PLO_E_RANGE (-3)    /* exact-integer magnitude bound exceeded (would overflow)   */
#define PLO_E_SHAPE (-4)    /* (m,k,n) shape / size not supported by the compiled kernels */
#define PLO_E_NODEVICE (-5) /* no CUDA device: there is NO CPU fallback                   */

#define PLO_MEASURE_NNZ 0 /* src/orbiter.cpp:146-153 Operations<0> + nonzeroes tie-break */
#define PLO_MEASURE_G2 3  /* src/growthfactor.cpp:117-125 G2                             */

#define PLO_MODE_EXHAUSTIVE 0 /* index is a mixed-radix code of the digits               */
#define PLO_MODE_PHILOX 1     /* digits drawn from Philox4x32-10(key=seed, ctr=index)    */

#define PLO_NO_INDEX UINT64_MAX

int plo_version(void);
int plo_device_count(void);           /* number of visible CUDA devices (0 => every call returns PLO_E_NODEVICE) */
int plo_set_device(int device);
const char* plo_last_error(void);     /* thread-local message of the last failing call */
void plo_release_workspace(void);     /* returns the cached device blocks of destroyed plans to the driver */
int plo_set_sweep_devices(int n);     /* host-level orbit sweeps (plo_orbiter) are sharded over the first n devices (default 1) */
/* 1: orbit shapes without a compiled kernel, and triples too large for the constant bank, run on the runtime-shape kernels (any
 * m, k, n <= 8; L | R | P^T from device memory when it does not fit the bank); 0 (default): they return PLO_E_SHAPE.  Process-wide and host-only (no device needed), like plo_set_sweep_devices: set it before the sweeps, from the
 * thread that drives them.  Any other value: PLO_E_ARG.  See the orbit section below. */
int plo_set_orbit_any_shape(int enable);

/* ---------------------------------------------------------------------------
 * Sparsifier candidate search.
 * Replaces ONE (block,num) step of the quad loop of localSparsifier
 *   include/plinopt_sparsify.inl:299-314   (for i,j,k,l in Coeffs^4, l fastest)
 * together with the per-candidate body testLinComb
 *   include/plinopt_sparsify.inl:166-197   (setRow+rank independence filter,
 *                                           v = TM^T.w, zero counts, strict
 *                                           lexicographic '>' acceptance).
 *
 * p == 0 : exact integers.  The caller pre-scales every COLUMN of TM by its LCD
 *          and coeffs by their common LCD (zero patterns of v = TM^T.w and of
 *          w are invariant under column / global scalings; rows of TM must NOT
 *          be scaled individually).  |values| must
 *          keep every v_j inside int64, else PLO_E_RANGE.
 * p  > 0 : residues mod p in [0,p), p < 2^32 (src/sparsifier.cpp:71-76).
 * TM       n x m row-major (n = TM.rowdim() = width of the CoB block).
 * off      4*block ; the candidate w has coeffs[i],[j],[k],[l] at positions
 *          off..off+3 (positions >= n are truncated, reference quirk Q4).
 * coeffs   c values in the reference's enumeration order (c <= 511: every index < c^4 has its own 36-bit key field below the
 *          seed's).
 * prev_rows nprev x n : the rows of LCoB chosen so far (Cand rows 0..num-1,
 *          plinopt_sparsify.inl:289,172); a candidate is admissible iff it is
 *          linearly independent of them (rank(Cand) > num, :173-175).
 * init_rl/init_cl  the weight seed (:290-295): (-1,-1) or the nullspace seed.
 * Outputs: the weight after the loop and the index ((i*c+j)*c+k)*c+l of the
 * accepted candidate = the FIRST maximiser in enumeration order (:183-184);
 * *best_index == PLO_NO_INDEX if no candidate beat the seed.
 * ------------------------------------------------------------------------ */
int plo_lincomb_search(uint32_t p, int n, int m, const int64_t* TM, int off, int c, const int64_t* coeffs,
                       int nprev, const int64_t* prev_rows, int init_rl, int init_cl,
                       int* best_rl, int* best_cl, uint64_t* best_index);

/* Same search for `nbatch` independent problems in one launch sequence (the
 * independent column blocks of blockSparsifier, plinopt_sparsify.inl:710-723):
 * problem b uses TM + b*n*m, coeffs + b*c, prev_rows + b*nprev*n, init_*[b]. */
int plo_lincomb_search_batch(uint32_t p, int nbatch, int n, int m, const int64_t* TM, int off, int c,
                             const int64_t* coeffs, int nprev, const int64_t* prev_rows, const int* init_rl,
                             const int* init_cl, int* best_rl, int* best_cl, uint64_t* best_index);

/* ALL the rows of one inner block in one launch sequence ("score once, filter four times").
 * In include/plinopt_sparsify.inl:282-326 the quad loop runs once per row num = 0..3 of an inner block, but the score
 * (rlHw, clHw) of a candidate (:176-180) does not depend on num; only the independence filter (:172-175) and the weight seed
 * (:290-295) do.  plo_lincomb_quad scores every candidate ONCE on the device and then picks the rows one after the other, the
 * filter of row num being derived on the device from the winners of rows 0..num-1: one host->device copy, six kernel launches
 * and one device->host copy for any number of independent problems (the column blocks of blockSparsifier, :710-723).
 * The rows are exactly those of successive plo_lincomb_search calls for the rows nprev .. off+3 of the block (min(4, n - off)
 * rows when nprev <= off; fewer when the call resumes inside a block), each with the previous winners appended to prev_rows
 * and, after the first, the weight seed (-1, -1).
 *
 * Per problem (m, the number of columns of TM, is common to the call, m <= 64; sum of c^4 <= PLO_QUAD_MAX_COUNT_BYTES):
 *   n, off, c, nprev, TM, coeffs, prev_rows, init_rl, init_cl   as in plo_lincomb_search (seed of the FIRST row);
 *   seed_vec  (n entries, scaled like prev_rows, or NULL) the vector that holds the seed weight -- the nullspace vector of
 *             :227-252; when it keeps row 0 and lives on the positions off..off+3 the device goes on with it as a previous row.
 * Outputs: rl/cl/index[t] for the rows t < nrows that were decided (index == PLO_NO_INDEX: the seed vector kept row 0), and
 *   status  PLO_QUAD_DONE   all the rows of the block decided;
 *           PLO_QUAD_MISS   row `nrows` has no admissible candidate: the caller applies the canonical fallback (:317-326)
 *                           and calls again for the remaining rows;
 *           PLO_QUAD_SEED   the seed vector kept row 0 and the device could not go on with it (seed_vec NULL or not on the
 *                           live positions): nrows == 1, call again with it among prev_rows;
 *           PLO_QUAD_RANGE  the exact-integer guard of the device-side filter tripped at row `nrows`: go on with
 *                           plo_lincomb_search for that row (never a silent wrap-around).  Over Q this is also the status,
 *                           with nrows == 0, of a problem whose prev_rows give annihilator functionals too large for the
 *                           device-side filter; the other problems of the call are decided as usual. */
#define PLO_QUAD_DONE 0
#define PLO_QUAD_MISS 1
#define PLO_QUAD_SEED 2
#define PLO_QUAD_RANGE 3
#define PLO_QUAD_MAX_COUNT_BYTES (1ull << 31)
typedef struct plo_quad_problem {
  int n, off, c, nprev;
  const int64_t* TM;        /* n x m */
  const int64_t* coeffs;    /* c */
  const int64_t* prev_rows; /* nprev x n */
  const int64_t* seed_vec;  /* n, may be NULL */
  int init_rl, init_cl;
  int nrows, status;        /* out */
  int rl[4], cl[4];         /* out */
  uint64_t index[4];        /* out */
} plo_quad_problem;
int plo_lincomb_quad(uint32_t p, int m, int nproblems, plo_quad_problem* problems);

/* Device-resident variant used for throughput measurement: inputs are uploaded
 * once, every plo_lincomb_plan_run() enqueues one full search on `stream`
 * (a cudaStream_t passed as void*, NULL = default stream). */
typedef struct plo_lincomb_plan plo_lincomb_plan;
int plo_lincomb_plan_create(plo_lincomb_plan** plan, uint32_t p, int nbatch, int n, int m, const int64_t* TM, int off,
                            int c, const int64_t* coeffs, int nprev, const int64_t* prev_rows, const int* init_rl,
                            const int* init_cl);
int plo_lincomb_plan_run(plo_lincomb_plan* plan, void* stream);
/* The same restricted to the candidates whose prefix (i*c+j)*c+k lies in [prefix_lo, prefix_hi): one GPU's share of a
 * search sharded over several devices (the partial winners are merged by the caller: lexicographic maximum of
 * (rl, cl, -index)). */
int plo_lincomb_plan_run_range(plo_lincomb_plan* plan, uint64_t prefix_lo, uint64_t prefix_hi, void* stream);
int plo_lincomb_plan_result(plo_lincomb_plan* plan, void* stream, int* best_rl, int* best_cl, uint64_t* best_index);
uint64_t plo_lincomb_plan_candidates(const plo_lincomb_plan* plan); /* candidates scored per run            */
int plo_lincomb_plan_launches(const plo_lincomb_plan* plan);         /* kernel launches per run              */
void plo_lincomb_plan_destroy(plo_lincomb_plan* plan);

/* ---------------------------------------------------------------------------
 * DeGroote-orbit sweep.
 * Replaces the whole `omp parallel for` + `omp critical` loop of
 *   src/orbiter.cpp:272-324
 * i.e. per candidate: zoiRandomMatrix x3 (:59-75,125-136), inverse /
 * inverseTranspose (plinopt_sparsify.inl:380-465), Tensor
 * (plinopt_library.inl:210-223), the three products (:288-294), the measure
 * (density/nonzeroes plinopt_library.inl:238-284, or G2 growthfactor.cpp:117-125)
 * and the keep-best rule (:298-323, made deterministic: lexicographic minimum,
 * lowest index among ties).
 *
 * L  r x (m*k), R  r x (k*n), P  (m*n) x r, row-major, entries pre-scaled to
 * integers: true matrix = L/denL etc. (p == 0), or residues in [0,p) with the
 * denominators ignored (2 <= p < 2^31: `orbiter -m p`, the search runs in Z/pZ,
 * src/orbiter.cpp:232-234,419-426; sparsity measure only).  Candidate `index` in [lo,hi) is decoded to (U,V,W) by the
 * counter-based decode documented in DESIGN.md (identical on host and device,
 * see plo_orbit_decode).
 *
 * Shapes: 2x2x2, 3x3x3, 4x4x4, 3x4x7, 3x3x6, 3x6x3 and 6x3x3 have compiled kernels; any other shape returns PLO_E_SHAPE unless
 * plo_set_orbit_any_shape(1) is in effect, which sends it, through every entry point below (plans, tables, survivors, 64-bit,
 * Z/pZ) and plo_orbiter*, to the runtime-shape kernels (DESIGN.md 5.1): one candidate per thread, int64 arithmetic, same decode,
 * same measures, same deterministic winner.  L | R | P^T is read from the constant bank when r.(mk+kn+mn) <= 12000 ints (6000
 * for the 64-bit entry points), else from device memory (kernel "orbit_rt_kernel+global"); that holds for the compiled shapes too.
 * Their limits, each PLO_E_SHAPE with its own message: m, k, n <= 8; at most 2^24 ints of L | R | P^T (2^23 for the 64-bit entry
 * points); exhaustive mode needs plo_orbit_space != 0.  With the switch at 0 a triple beyond the bank is PLO_E_SHAPE.
 * A compiled shape whose triple fits the bank keeps its kernel whatever the switch; PLO_ORBIT_RUNTIME_SHAPE set in the
 * environment sends it to the runtime-shape kernels as well (A/B timing and parity only: identical results, except that G2 on the 64-bit paths -- beyond the
 * int32 magnitude bound or through plo_orbit_sweep64 / table64 -- may differ from orbit_wide_kernel in the last bits).
 * ------------------------------------------------------------------------ */
typedef struct plo_orbit_best {
  double score;   /* measure 0: (double)nnz ; measure 3: G2                    */
  uint32_t nnz;   /* nnz(Lj)+nnz(Rg)+nnz(hP)      (plinopt_library.inl:279-284) */
  uint32_t nno;   /* entries not in {0,+1,-1}                                   */
  uint64_t index; /* winning candidate, PLO_NO_INDEX if lo >= hi                */
} plo_orbit_best;

int plo_orbit_sweep(uint32_t p, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P,
                    int32_t denL, int32_t denR, int32_t denP, int measure, int mode, uint64_t seed, uint64_t lo,
                    uint64_t hi, plo_orbit_best* best);

/* The exact sweep sharded over the first `ndev` CUDA devices of the calling process (clamped to the devices present): contiguous
 * ascending index shards, asynchronous launches from one host thread, same winner as the single-device call.  This is what
 * `bin/orbiter --gpus N` uses; multi-process runs shard with plo_orbit_plan_run + one all-reduce instead (INTEGRATION.md). */
int plo_orbit_sweep_devices(int ndev, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P,
                            int32_t denL, int32_t denR, int32_t denP, int measure, int mode, uint64_t seed, uint64_t lo,
                            uint64_t hi, plo_orbit_best* best);

/* index -> (U,V,W), row-major int32 in {-1,0,1}; pure host function, bit-identical to the device decode. */
int plo_orbit_decode(int m, int k, int n, int mode, uint64_t seed, uint64_t index, int32_t* U, int32_t* V, int32_t* W);
/* size of the exhaustive candidate space (0 if it does not fit in 64 bits) */
uint64_t plo_orbit_space(int m, int k, int n);

/* Per-candidate table (nnz, nno, g2) for [lo,hi): parity / debugging; any output may be NULL. */
int plo_orbit_table(int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int32_t denL,
                    int32_t denR, int32_t denP, int mode, uint64_t seed, uint64_t lo, uint64_t hi, uint32_t* nnz,
                    uint32_t* nno, double* g2);

/* 64-bit inputs: entries and common denominators beyond the int32 C ABI above (2x2x2_7_DPS-intermediate-12.0695 has a common
 * denominator of 1.0e11); |entries| < 2^46; every compiled shape; same decode, same deterministic winner; G2 within 1e-12
 * relative of growthfactor.cpp:117-125.  Synchronous. */
int plo_orbit_sweep64(int m, int k, int n, int r, const int64_t* L, const int64_t* R, const int64_t* P, int64_t denL, int64_t denR,
                      int64_t denP, int measure, int mode, uint64_t seed, uint64_t lo, uint64_t hi, plo_orbit_best* best);
int plo_orbit_table64(int m, int k, int n, int r, const int64_t* L, const int64_t* R, const int64_t* P, int64_t denL, int64_t denR,
                      int64_t denP, int mode, uint64_t seed, uint64_t lo, uint64_t hi, uint32_t* nnz, uint32_t* nno, double* g2);

/* The same table over Z/pZ (residues in, (nnz, nno) per candidate out). */
int plo_orbit_table_modp(uint32_t p, int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int mode,
                         uint64_t seed, uint64_t lo, uint64_t hi, uint32_t* nnz, uint32_t* nno);

/* Device-resident plan (throughput measurement / multi-GPU sharding). */
typedef struct plo_orbit_plan plo_orbit_plan;
int plo_orbit_plan_create(plo_orbit_plan** plan, int m, int k, int n, int r, const int32_t* L, const int32_t* R,
                          const int32_t* P, int32_t denL, int32_t denR, int32_t denP, int measure, int mode,
                          uint64_t seed);
int plo_orbit_plan_run(plo_orbit_plan* plan, uint64_t lo, uint64_t hi, void* stream);
int plo_orbit_plan_result(plo_orbit_plan* plan, void* stream, plo_orbit_best* best);
int plo_orbit_plan_launches(const plo_orbit_plan* plan);
/* Multi-GPU plumbing without a host hop (the reference analogue is the `omp critical` of src/orbiter.cpp:298): writes the winner of
 * the last run on `stream` into slot `rank` of a DEVICE table of world x 4 int64 words (order-preserving bits of the score, index,
 * nnz, nno; INT64_MAX elsewhere).  One all-reduce(MIN) over the table (ncclAllReduce / torch.distributed on the same buffer)
 * then leaves every local winner on every rank; the global one is the lexicographic minimum of (score[, nno], index). */
int plo_orbit_plan_pack(plo_orbit_plan* plan, int64_t* slots_device, int rank, int world, void* stream);
/* Name of the sweep kernel plo_orbit_plan_run launches for this plan and the number of candidate-matrix entries one 32-bit
 * multiply-add carries in it (1 scalar, 2 sixteen-bit lanes, 4 eight-bit lanes): the roofline of a sweep is stated against
 * lanes x the measured IMAD peak, and a profile is only quoted for the kernel it was taken from. */
int plo_orbit_plan_kernel(const plo_orbit_plan* plan, char* name, int cap, int* lanes);
/* Host-only (no device needed): the worst-case magnitudes of the transformed entries of L.(U^-1 (x) V), R.(V^-T (x) W),
 * (U (x) W^-1).P over the whole orbit, bounds[3], that select the lane packing.  Returns 4 / 2 / 1 (eight-bit lanes, sixteen-bit
 * lanes, scalar int32 kernel) or 0 (beyond the int32 product bound: 64-bit kernels), PLO_E_ARG on bad arguments. */
int plo_orbit_magnitude_bounds(int m, int k, int n, int r, const int32_t* L, const int32_t* R, const int32_t* P, int64_t* bounds);
/* Host-only self-test (no device needed) of the whole-matrix decode behind the table-driven 2x2x2 kernels: number of mismatches
 * between digit-by-digit decoding and replaying matrix number floor(x.count/2^32) resp. rem mod count; 0 = consistent. */
int plo_selftest_matrix_index(void);
/* Survivor compaction (north_star: "surviving candidates are compacted through coalesced vectorised stores"): every candidate of
 * [lo,hi) whose score does not exceed `threshold` -- sparsity plans: (nnz, nno) <= (threshold->nnz, threshold->nno)
 * lexicographically (the order of src/orbiter.cpp:300-312); growth-factor plans: G2 <= threshold->score -- is returned with BOTH
 * measures (nnz, nno, score = growth factor), sorted by index.  Synchronous.  *count = survivors found; if that exceeds `capacity`
 * nothing is written and PLO_E_RANGE is returned (call again with room for *count records or a tighter threshold). */
int plo_orbit_plan_survivors(plo_orbit_plan* plan, uint64_t lo, uint64_t hi, const plo_orbit_best* threshold, uint64_t capacity,
                             plo_orbit_best* out, uint64_t* count);
void plo_orbit_plan_destroy(plo_orbit_plan* plan);

/* Orbit sweeps over Q(sqrt d), d an integer that is not a perfect square (the reference's `-P "X^2-d"`; DESIGN.md 5.1).  Every
 * entry is (a + b.sqrt(d)) / den: La, Ra, Pa hold the integers a, Lb, Rb, Pb the integers b, in the layout of plo_orbit_plan_create,
 * with one common denominator per matrix.  An entry is zero iff a = b = 0 and +-1 iff b = 0 and a = +-den; G2 takes the real
 * embedding sqrt(d) > 0 and converts every entry to a double before squaring, so it exists for d > 0 only.  Any shape up to 8x8x8
 * runs on the runtime-shape kernel, compiled shapes included, whatever plo_set_orbit_any_shape says.  The host stores the entries as
 * int32 when they all fit, else as int64.  run, result, pack, survivors, kernel ("orbit_rt_kernel+quad", 1 lane) and destroy work on
 * the plan as on any other.  Both parts go to the constant bank when 2.r.(mk+kn+mn) <= 12000 ints (4.r.(mk+kn+mn) for int64
 * storage); beyond it, with plo_set_orbit_any_shape(1), to device memory ("orbit_rt_kernel+quad+global"), up to 2^24 ints, else
 * PLO_E_SHAPE; |entries| < 2^53 and every transformed entry of each part below 2^62 (PLO_E_RANGE); d a perfect square,
 * or measure G2 with d < 0 (PLO_E_ARG). */
int plo_orbit_plan_create_quad(plo_orbit_plan** plan, int64_t d, int m, int k, int n, int r, const int64_t* La, const int64_t* Lb,
                               const int64_t* Ra, const int64_t* Rb, const int64_t* Pa, const int64_t* Pb, int64_t denL, int64_t denR,
                               int64_t denP, int measure, int mode, uint64_t seed);
/* Per-candidate (nnz, nno, g2) of [lo,hi) over Q(sqrt d); any output may be NULL, g2 must be NULL when d < 0. */
int plo_orbit_table_quad(int64_t d, int m, int k, int n, int r, const int64_t* La, const int64_t* Lb, const int64_t* Ra, const int64_t* Rb,
                         const int64_t* Pa, const int64_t* Pb, int64_t denL, int64_t denR, int64_t denP, int mode, uint64_t seed, uint64_t lo,
                         uint64_t hi, uint32_t* nnz, uint32_t* nno, double* g2);

/* ---------------------------------------------------------------------------
 * Growth factor G2 of explicit triples  (src/growthfactor.cpp:117-125, rows
 * converted to double before squaring :25-28,41-44).  Dense double inputs,
 * `batch` triples stored back to back; out[b] = sum_i |L_i| |R_i| |P^T_i|.
 * ------------------------------------------------------------------------ */
int plo_growth_G2(int batch, int r, int a, int b, int c, const double* L, const double* R, const double* P, double* out);

/* ---------------------------------------------------------------------------
 * Batched MMchecker mod p.
 * Replaces PLinOpt::MMchecker  include/plinopt_library.inl:472-558 for `batch`
 * independent random evaluations: wc = P.((L.ua) o (R.ub)) against the direct
 * product reshape(ua).reshape(ub)  (:504-528).
 * CSR inputs with residues in [0,p), p < 2^32 odd or 2 (src/MMchecker.cpp:123-126).
 * ua (batch x m*k) / ub (batch x k*n) may be NULL: then they are Philox words
 * mod p drawn from (seed, sample index).  ok[s] = 1 iff sample s agrees.
 * Returns 0 (all samples agree: "correct"), 1 (some sample disagrees: not an MM
 * algorithm, :555), 3 (outer dimension mismatch, :494) or PLO_E_*.
 * ------------------------------------------------------------------------ */
typedef struct plo_csr {
  int rows, cols;
  const int64_t* ptr;  /* rows+1 */
  const int32_t* col;  /* nnz    */
  const uint32_t* val; /* nnz residues */
} plo_csr;

int plo_mmcheck_batch(uint32_t p, int m, int k, int n, int r, const plo_csr* L, const plo_csr* R, const plo_csr* P,
                      uint64_t seed, int batch, const uint32_t* ua, const uint32_t* ub, uint8_t* ok);

typedef struct plo_mmcheck_plan plo_mmcheck_plan;
int plo_mmcheck_plan_create(plo_mmcheck_plan** plan, uint32_t p, int m, int k, int n, int r, const plo_csr* L,
                            const plo_csr* R, const plo_csr* P, int batch);
int plo_mmcheck_plan_run(plo_mmcheck_plan* plan, uint64_t seed, uint64_t first_sample, void* stream);
int plo_mmcheck_plan_result(plo_mmcheck_plan* plan, void* stream, uint8_t* ok, int* verdict);
int plo_mmcheck_plan_launches(const plo_mmcheck_plan* plan);
/* What the encoder made of L, R, P (each array may be NULL): loads[3] = X words read per sample (the CSR has nnz of them),
 * blob_bytes[3] = size of the encoded matrix, strides[6] = (column stride of the column block sums, row stride of the row block
 * sums) per matrix, 0 = not used. */
int plo_mmcheck_plan_encoding(const plo_mmcheck_plan* plan, int64_t* loads, int64_t* blob_bytes, int* strides);
/* The random coordinates plo_mmcheck_plan_run draws are (Philox word & (2^bits - 1)) mod p, bits = 1..32 (default 32): the same
 * integer point under every modulus, which is what lets plo_mmchecker decide equality over Q from several primes. */
int plo_mmcheck_plan_input_bits(plo_mmcheck_plan* plan, int bits);
void plo_mmcheck_plan_destroy(plo_mmcheck_plan* plan);
/* Host-only check (no device needed) of the matrix encoder behind the plans: encodes A the way plan_create does for `groups`
 * sample groups (column block sums; when row_blocks != 0 also row block sums and outputs numbered by task with fold lists, the
 * way plans encode P; plain pairs and value groups; see csrc/mmcheck.cu), replays the encoded stream on the CPU for ONE sample and returns y = A.x mod p (x: cols residues,
 * y: rows).  stats (may be NULL, 9 values): row stride of the row blocks (0: none), column stride of the column blocks (0: none),
 * chunks, blob bytes, plain entries, units of 4 grouped entries, value groups, X loads per sample after encoding, stored
 * (row, slab) tasks. */
int plo_mmcheck_encode_check(uint32_t p, const plo_csr* A, int groups, int row_blocks, const uint32_t* x, uint32_t* y, long long* stats);

/* ---------------------------------------------------------------------------
 * Factorizer random restarts  (SURVEY.md section 8 row f2).
 * Replaces the `omp parallel for` over `randomloops` calls of backSolver in
 * PLinOpt::Factorizer  include/plinopt_sparsify.inl:960-985  (backSolver :755-867,
 * order tricOpCount :914-921).  Candidate `index` = one random row order of M
 * (plo_factor_decode); its score is (nnz(Alt), #entries of Alt not in {0,+-1},
 * nnz(CoB)) of the factorisation M = Alt.CoB that backSolver builds from that
 * order, inner dimension k (n <= k <= r).  M: r x n residues mod an odd prime
 * p < 2^31, 1 <= n <= 64, r <= 512, full column rank (candidates whose first
 * rows never reach rank n score as "none"); other shapes: PLO_E_ARG.  The plan
 * picks the kernel from the shape: factor_sweep_kernel for n <= 32 and r <= 255,
 * factor_wide_kernel for the rest; both score the same candidates.
 * Lexicographic minimum, lowest index among ties.
 * table (may be NULL): 3 x (hi-lo) words (nnz_alt, nno_alt, nnz_cob) per candidate.
 * ------------------------------------------------------------------------ */
typedef struct plo_factor_best {
  uint32_t nnz_alt, nno_alt, nnz_cob, pad_;
  uint64_t index; /* PLO_NO_INDEX if no candidate */
} plo_factor_best;

int plo_factor_sweep(uint32_t p, int r, int n, int k, const uint32_t* M, uint64_t seed, uint64_t lo, uint64_t hi,
                     plo_factor_best* best, uint32_t* table);
/* perm[t] = original row standing at position t of candidate `index` (host function, same digits as the device) */
int plo_factor_decode(int r, uint64_t seed, uint64_t index, int32_t* perm);

typedef struct plo_factor_plan plo_factor_plan;
int plo_factor_plan_create(plo_factor_plan** plan, uint32_t p, int r, int n, int k, const uint32_t* M, uint64_t seed);
int plo_factor_plan_run(plo_factor_plan* plan, uint64_t lo, uint64_t hi, void* stream);
int plo_factor_plan_result(plo_factor_plan* plan, void* stream, plo_factor_best* best);
int plo_factor_plan_launches(const plo_factor_plan* plan);
/* name of the kernel the plan launches, e.g. "factor_sweep_kernel<16>" or "factor_wide_kernel<2>" (NUL-terminated, cap bytes) */
int plo_factor_plan_kernel(const plo_factor_plan* plan, char* name, int cap);
void plo_factor_plan_destroy(plo_factor_plan* plan);

/* ---------------------------------------------------------------------------
 * dependency `Explore`  (SURVEY.md section 8 row f3).
 * Replaces the recursive enumeration of src/dependency.cpp:73-100 (driver Depender :106-169):
 * for every start row i and every choice of 1 <= d <= level-1 further rows i < q_1 < .. < q_d with
 * coefficients C[v_1..v_d], test W = base[i] + sum_t prod[q_t][v_t] for being zero (pos = -1) or having
 * exactly one non-zero coordinate (pos = that coordinate).  base (r x n) = the rows of M, prod
 * (r x c x n) = C[v].M[q], both in the field: residues mod p (p > 0) or integers scaled by a common
 * denominator (p == 0, |entries| <= 2^60).  Hits come back in the reference's depth-first order
 * (a combination before its extensions); *nhits is the total found, *ncand the number of combinations tested.  When more hits
 * exist than max_hits the call returns PLO_E_RANGE with *nhits set (call again with room for all of them): the records stored in
 * that case are an arbitrary subset, not the first lines of the reference's output.
 * ------------------------------------------------------------------------ */
typedef struct plo_dep_hit {
  int32_t depth;    /* number of added rows d */
  int32_t pos;      /* -1: zero vector; else the single non-zero coordinate */
  int32_t rows[5];  /* i, q_1 .. q_d ; -1 beyond */
  int32_t coefs[5]; /* -1 (the start row has coefficient one), v_1 .. v_d ; -1 beyond */
} plo_dep_hit;

int plo_dependency_explore(uint32_t p, int r, int n, int c, int level, const int64_t* base, const int64_t* prod,
                           uint64_t max_hits, plo_dep_hit* hits, uint64_t* nhits, uint64_t* ncand);

/* ---------------------------------------------------------------------------
 * The one collective of the path, issued by the engine: an all-reduce (min / max) over a few int64 words of device memory through
 * NCCL (one rank per GPU and process).  north_star: "a single tiny NCCL allreduce(min-with-index) picks the global best"; reference
 * analogue: the `omp critical` of src/orbiter.cpp:298.  NCCL is bound at run time (dlopen of libnccl.so.2), so single-GPU users
 * never need it.  Rank 0 calls plo_comm_unique_id and hands the 128 bytes to the other ranks through whatever launched them
 * (bench.py: torch.distributed broadcast); every rank then calls plo_comm_create on its own device.  A sweep step on N GPUs is
 *   plo_orbit_plan_run -> plo_orbit_plan_pack(slots) -> plo_comm_allreduce_i64(slots, 4*N, PLO_REDUCE_MIN)   all on one stream,
 * the sparsifier search merges its packed (rl, cl, -index) keys with PLO_REDUCE_MAX.
 * ------------------------------------------------------------------------ */
#define PLO_REDUCE_MIN 0
#define PLO_REDUCE_MAX 1
typedef struct plo_comm plo_comm;
int plo_comm_nccl_version(void);                 /* 0 when libnccl.so.2 cannot be loaded */
int plo_comm_unique_id(uint8_t* id128);          /* 128 bytes, rank 0 */
int plo_comm_create(plo_comm** comm, int rank, int world, const uint8_t* id128);
int plo_comm_rank(const plo_comm* comm);
int plo_comm_size(const plo_comm* comm);
int plo_comm_allreduce_i64(plo_comm* comm, int64_t* buf_device, uint64_t count, int op, void* stream);  /* in place, asynchronous on `stream` */
void plo_comm_destroy(plo_comm* comm);

/* ---------------------------------------------------------------------------
 * The other sweeps sharded over the first `ndev` CUDA devices of the calling process (clamped to the devices present), like
 * plo_orbit_sweep_devices: one host thread, asynchronous launches, results merged in device order -- same answers as the
 * single-device calls.  Reference analogues: the omp loops of include/plinopt_sparsify.inl:962,968 and src/orbiter.cpp:272.
 *   plo_lincomb_search_devices  one (batched) sparsifier search, the prefix range (i*c+j)*c+k split over the devices
 *   plo_mmcheck_batch_devices   `batch` Philox samples split over the devices (ok[s] as in plo_mmcheck_batch; returns its verdict)
 *   plo_factor_sweep_devices    Factorizer random restarts [lo,hi) split over the devices
 * ------------------------------------------------------------------------ */
int plo_lincomb_search_devices(int ndev, uint32_t p, int nbatch, int n, int m, const int64_t* TM, int off, int c, const int64_t* coeffs,
                               int nprev, const int64_t* prev_rows, const int* init_rl, const int* init_cl, int* best_rl, int* best_cl,
                               uint64_t* best_index);
int plo_mmcheck_batch_devices(int ndev, uint32_t p, int m, int k, int n, int r, const plo_csr* L, const plo_csr* R, const plo_csr* P,
                              uint64_t seed, int batch, uint8_t* ok);
int plo_factor_sweep_devices(int ndev, uint32_t p, int r, int n, int k, const uint32_t* M, uint64_t seed, uint64_t lo, uint64_t hi,
                             plo_factor_best* best);

/* ---------------------------------------------------------------------------
 * Roofline denominators that MEASURED_PEAKS.json does not hold: register-
 * resident unrolled IMAD / DFMA / (ISETP+IADD) loops over all SMs, CUDA-event
 * timed, best of `reps`.  Results in operations per second.
 * ------------------------------------------------------------------------ */
int plo_measure_peaks(int reps, double* imad_per_s, double* dfma_per_s, double* ialu_per_s);
/* Scheduler issue peak: IMAD (fma-heavy pipe) and LOP3 (alu pipe) chains interleaved one to one; thread instructions per
 * second (= SMs x 4 schedulers x 32 lanes x clock when both pipes are kept full). */
int plo_measure_issue_peak(int reps, double* inst_per_s);

/* ---------------------------------------------------------------------------
 * Host-level entry points (C++ host orchestration around the kernels above;
 * plinopt_b200/csrc/host/).  Rationals cross the boundary as (num, den) int64
 * arrays, row-major.
 * ------------------------------------------------------------------------ */

/* blockSparsifier  include/plinopt_sparsify.inl:666-748  as driven by TSparsifier
 * src/sparsifier.cpp:20-55: M (rows x cols) -> CoB (cols x cols), Res (rows x cols) with
 * M == Res.CoB (consistency(), :871-907, reported in *consistent).  q == 0: over Q; q > 0: over
 * Z/qZ (entries a/b -> a.b^-1 mod q, src/sparsifier.cpp:71-76; outputs are residues with den 1).
 * stats (may be NULL): [0] candidates scored on the GPU, [1] GPU searches, [2] canonical fallbacks.
 * log_fd: file descriptor for the reference's '# [SPRF] ...' progress lines (-1: silent). */
int plo_sparsifier(uint64_t q, int rows, int cols, const int64_t* num, const int64_t* den, int blocksize,
                   int maxnumcoeff, int initialElimination, int64_t* cob_num, int64_t* cob_den,
                   int64_t* res_num, int64_t* res_den, int* consistent, uint64_t* stats, int log_fd);

/* Orbiter<Measure>::operator()  src/orbiter.cpp:215-360  over Q: sweeps candidates [0, loops),
 * applies the acceptance rule against the input (:330-331) and, if the winner improves on it,
 * returns the transformed triple (exact rationals) and re-checks it with MMchecker (:355). */
typedef struct plo_orbiter_report {
  uint32_t init_nnz, init_nno;
  double init_score;
  plo_orbit_best best;
  int improved;    /* 1: outputs hold the transformed triple, 0: outputs hold the input */
  int mm_verdict;  /* MMchecker verdict of the returned triple (0 = correct) */
  int m, k, n;
} plo_orbiter_report;

int plo_orbiter(int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd, const int64_t* Pn,
                const int64_t* Pd, int64_t* oLn, int64_t* oLd, int64_t* oRn, int64_t* oRd, int64_t* oPn, int64_t* oPd,
                plo_orbiter_report* report);

/* The '# Found opt:' records of src/orbiter.cpp:300-318, deterministic: the reference prints every candidate that improves on the
 * best so far as its OpenMP threads meet them; in index order those are the successive minima of the prefixes [0, i] that also
 * improve on the input triple (acceptance :300-302).  records[0..*count) in increasing index order, the last one being the winner
 * plo_orbiter returns; PLO_E_RANGE (with *count set) when `capacity` is too small.  Costs about one more sweep. */
int plo_orbiter_progress(int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                         const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd, const int64_t* Pn,
                         const int64_t* Pd, uint64_t capacity, plo_orbit_best* records, uint64_t* count);

/* plo_orbiter and plo_orbiter_progress over Q(sqrt d), d an integer that is not a perfect square (`orbiter -P "X^2-d"`).  Each
 * matrix comes as four arrays (an, ad, bn, bd), entry an/ad + bn/bd.sqrt(d) (NULL denominators: 1); the outputs use the same
 * layout.  The sweep runs on plo_orbit_plan_create_quad plans with one common denominator per matrix over both parts, sharded over
 * the devices of plo_set_sweep_devices; an entry is zero iff both parts are zero and +-1 iff bn = 0 and an/ad = +-1.  The winner is
 * accepted as over Q, its transform is exact (each part separately) and mm_verdict comes from plo_mmchecker_quad.  Limits of
 * plo_orbit_plan_create_quad; G2 needs d > 0 (PLO_E_ARG). */
int plo_orbiter_quad(int64_t d, int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                     const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn, const int64_t* Lbd, const int64_t* Ran, const int64_t* Rad,
                     const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan, const int64_t* Pad, const int64_t* Pbn, const int64_t* Pbd,
                     int64_t* oLan, int64_t* oLad, int64_t* oLbn, int64_t* oLbd, int64_t* oRan, int64_t* oRad, int64_t* oRbn, int64_t* oRbd,
                     int64_t* oPan, int64_t* oPad, int64_t* oPbn, int64_t* oPbd, plo_orbiter_report* report);
int plo_orbiter_progress_quad(int64_t d, int measure, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                              const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn, const int64_t* Lbd, const int64_t* Ran,
                              const int64_t* Rad, const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan, const int64_t* Pad,
                              const int64_t* Pbn, const int64_t* Pbd, uint64_t capacity, plo_orbit_best* records, uint64_t* count);

/* fMMchecker + MMchecker  src/MMchecker.cpp:48-81, include/plinopt_library.inl:472-558 on dense
 * rational inputs, `batch` independent random evaluations.
 * modulus > 0: in Z/pZ, p = modulus without its factors of 2 (:123-126).
 * modulus == 0: over Q.  The reference evaluates both sides exactly at a random point with `bitsize`-bit integer coordinates
 * (:497-528); this engine takes the same decision from residues: with D a common multiple of all denominators,
 * N = D.(P.((L.ua) o (R.ub)) - ua.ub) is an integer vector of known size bound, and the samples are checked modulo as many
 * word-size primes (2^31-1 downwards, skipping primes that divide a denominator) as it takes for their product to exceed 2|N|:
 * verdict 0 means both sides are EQUAL OVER Q at every sampled point, verdict 1 that they differ at one of them.
 * plo_mmchecker uses 32-bit coordinates; plo_mmchecker_bits takes the bit size (1..32, larger values are clamped; the reference's
 * `-b`) and reports the number of primes it used (*nprimes, may be NULL).
 * Returns 0 correct / 1 not an MM algorithm / 2 inner / 3 outer dimension mismatch / PLO_E_*. */
int plo_mmchecker(uint64_t modulus, uint64_t seed, int batch, int Lrows, int Lcols, int Rrows, int Rcols, int Prows,
                  int Pcols, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                  const int64_t* Pn, const int64_t* Pd, uint32_t* nnz_nno /* [2], may be NULL */);
int plo_mmchecker_bits(uint64_t modulus, int bitsize, uint64_t seed, int batch, int Lrows, int Lcols, int Rrows, int Rcols, int Prows,
                       int Pcols, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd,
                       const int64_t* Pn, const int64_t* Pd, uint32_t* nnz_nno /* [2], may be NULL */, int* nprimes);
/* The same check over Q(sqrt d), d an integer that is not a perfect square (`MMchecker -P "X^2-d"`), d < 0 allowed: each matrix
 * as (an, ad, bn, bd), entry an/ad + bn/bd.sqrt(d), NULL denominators 1.  The decision is exact at the sampled integer points:
 * only primes p (2^31-1 downwards) with d a non-zero square mod p and no vanishing denominator are used, each under both
 * embeddings sqrt(d) -> s and -s (s^2 = d mod p), with the same points; the size bound is that of the check over Q with
 * |a + b.sqrt d| = |a| + |b|.sqrt|d|.  nnz_nno counts as plo_orbiter_quad; *nprimes counts primes.  Same return codes;
 * PLO_E_ARG when d is a perfect square. */
int plo_mmchecker_quad(int64_t d, int bitsize, uint64_t seed, int batch, int Lrows, int Lcols, int Rrows, int Rcols, int Prows, int Pcols,
                       const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn, const int64_t* Lbd, const int64_t* Ran, const int64_t* Rad,
                       const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan, const int64_t* Pad, const int64_t* Pbn, const int64_t* Pbd,
                       uint32_t* nnz_nno /* [2], may be NULL */, int* nprimes);

/* The same over Z/qZ (`orbiter -m q`, src/orbiter.cpp:419-426): factors of 2 are stripped from q (:421-422), the
 * matrices are reduced first (:232-234), the search, the acceptance and the final MMchecker run in the field
 * (sparsity measure, Orbiter<0>).  Outputs are residues. */
int plo_orbiter_modp(uint64_t q, int mode, uint64_t seed, uint64_t loops, int r, int Lcols, int Rcols, int Prows,
                     const int64_t* Ln, const int64_t* Ld, const int64_t* Rn, const int64_t* Rd, const int64_t* Pn,
                     const int64_t* Pd, int64_t* oL, int64_t* oR, int64_t* oP, plo_orbiter_report* rep);

/* growthfactor  src/growthfactor.cpp:143-231: growth / error factors of one triple, in the reference's print order
 * out[11] = Ginfinf, Ginf2, G2inf, G22, G2, Q0, Qkinfinf, Q1inf2, Q12inf, Qk2inf, Q122.  G2 (:117-125, the measure the orbit sweep
 * minimises) is evaluated on the device; the other norms (:57-143) on the host. */
int plo_growth_factors(int r, int Lcols, int Rcols, int Prows, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn,
                       const int64_t* Rd, const int64_t* Pn, const int64_t* Pd, double* out);
/* The same eleven factors over Q(sqrt d), d > 0 and not a perfect square (`growthfactor -P "X^2-d"`): entry e of each matrix is
 * an[e]/ad[e] + bn[e]/bd[e].sqrt(d) (NULL denominators: 1), converted to a double with sqrt(d) > 0 before any norm. */
int plo_growth_factors_quad(int64_t d, int r, int Lcols, int Rcols, int Prows, const int64_t* Lan, const int64_t* Lad, const int64_t* Lbn,
                            const int64_t* Lbd, const int64_t* Ran, const int64_t* Rad, const int64_t* Rbn, const int64_t* Rbd, const int64_t* Pan,
                            const int64_t* Pad, const int64_t* Pbn, const int64_t* Pbd, double* out);

/* Factorizer  include/plinopt_sparsify.inl:924-990  (driver TFactorizer src/factorizer.cpp:28-97 without the
 * optional initial sparsification): M (rows x cols, full column rank) -> Alt (rows x k) . CoB (k x cols),
 * k = innerdim (0: cols), minimising (nnz(Alt), non-+-1 of Alt, nnz(CoB)) over `loops` random row orders
 * (candidates 0..loops-1 of plo_factor_sweep), starting from the trivial M = M.I (:958).  q == 0: over Q -- the
 * device scores candidates modulo a 31-bit prime, the winner is rebuilt exactly and its score verified;
 * q > 0: over Z/qZ.  Returns 0, -1 (inner dimension outside [cols, rows], :936-942) or PLO_E_*.
 * report (may be NULL, 8 words): initial (nnz, non-+-1, cols), final (nnz Alt, non-+-1 Alt, nnz CoB),
 * winning candidate (PLO_NO_INDEX: the trivial factorisation was kept), consistency M == Alt.CoB (:871-907). */
int plo_factorizer(uint64_t q, int rows, int cols, const int64_t* num, const int64_t* den, int innerdim, uint64_t loops,
                   uint64_t seed, int64_t* alt_num, int64_t* alt_den, int64_t* cob_num, int64_t* cob_den, uint64_t* report);

/* Depender  src/dependency.cpp:106-169: coefficient list ({1,-1} + user values + numerators and denominators of
 * the entries + 2,3,.., truncated to maxnumcoeff, images in the field, :118-146), then Explore (plo_dependency_explore)
 * with `level` monomials at most.  q == 0: over Q (exact, scaled integers); q > 0: over Z/qZ, q prime.
 * hits/nhits/ncand as in plo_dependency_explore; text (may be NULL): the reference's stdout, one line per stored hit
 * ("+o3-o5*2;" / "-i7+o3...;" showOut/showLC :47-71), NUL-terminated, *text_len = full length.
 * coef_num/coef_den (may be NULL, maxnumcoeff entries): the coefficient list used; *ncoef its length. */
int plo_depender(uint64_t q, int rows, int cols, const int64_t* num, const int64_t* den, int nuser, const int64_t* user_num,
                 const int64_t* user_den, int maxnumcoeff, int level, uint64_t max_hits, plo_dep_hit* hits, uint64_t* nhits,
                 uint64_t* ncand, char* text, uint64_t text_cap, uint64_t* text_len, int64_t* coef_num, int64_t* coef_den, int* ncoef);

/* negater  src/negater.cpp:117-209 (host only, exact over Q): per product i, the common divisors of the numerators and of the
 * denominators of row i of L and of R move into column i of P (unless only_sign), then two of (L_i, R_i, P^T_i) change sign when
 * that lowers the number of negative coefficients.  Outputs have the input shapes.  stats (may be NULL, 12 words): common
 * divisors before, after, rows flipped, negatives before in L,R,P, after in L,R,P, non-zeroes of L,R,P. */
int plo_negater(int only_sign, int r, int Lcols, int Rcols, int Prows, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn,
                const int64_t* Rd, const int64_t* Pn, const int64_t* Pd, int64_t* oLn, int64_t* oLd, int64_t* oRn, int64_t* oRd,
                int64_t* oPn, int64_t* oPd, uint64_t* stats);

/* rotater  bin/rotater.sh:75-83 (with src/columns-swap.cpp:41-52 and matrix-transpose): the cyclic rotation of an <m,k,n>
 * algorithm, left (right = 0): L' = R (r x kn), R' = (P^T)_s (r x nm), P' = (L_s)^T (km x r), an <k,n,m> algorithm; right:
 * L' = (P^T)_s (r x nm), R' = L (r x mk), P' = (R_s)^T (nk x r), an <n,m,k> algorithm.  Returns 3 on an outer dimension mismatch. */
int plo_rotater(int right, int r, int Lcols, int Rcols, int Prows, const int64_t* Ln, const int64_t* Ld, const int64_t* Rn,
                const int64_t* Rd, const int64_t* Pn, const int64_t* Pd, int64_t* oLn, int64_t* oLd, int64_t* oRn, int64_t* oRd,
                int64_t* oPn, int64_t* oPd);

/* Straight-line program -> matrix: matrixBuilder  include/plinopt_programs.inl:1459-1608 (with the
 * parser :618-686 and parenthesisExpand :1615-1679; driver src/SLPchecker.cpp:22-40, rule
 * data/Makefile:31-32).  Needed to regenerate data/32x32x32_15096_{L,R,P}.sms, which the reference
 * ships only as .slp (.MISSING_LARGE_BLOBS:1-3).  Two-step: build, then export into caller buffers
 * (CSR with rational values num/den). */
typedef struct plo_slp_matrix plo_slp_matrix;
int plo_slp_build(const char* text, char outchar, plo_slp_matrix** out, int* rows, int* cols, int64_t* nnz);
int plo_slp_export(const plo_slp_matrix* m, int64_t* ptr, int32_t* col, int64_t* num, int64_t* den);
void plo_slp_free(plo_slp_matrix* m);

/* include/plinopt_library.h:177-181 */
void plo_LRP2MM(int Lcols, int Rcols, int Prows, int* m, int* k, int* n);

#ifdef __cplusplus
}
#endif
#endif /* PLINOPT_B200_H */
