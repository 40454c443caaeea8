#!/usr/bin/env python3
"""Side benchmarks of the other two kernels of the hot path (not the bench.py headline):
  * sparsifier candidate search, BASELINE config 3 shape: 4x4x4_48_rational_L mod 2^31-1, 4 column
    blocks batched, c in {20, 64, 128}
  * batched MMchecker mod 2^31-1 on a synthetic CSR triple with the size/density of 32x32x32_15096
Prints one JSON line per case (CUDA-event timing on the launch stream, 3 warm-up runs)."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from plinopt_b200 import capi, hm  # noqa: E402

P31 = 2147483647
BATCHES = (32, 256, 1024, 4096)


def coeff_list(tm, p, c):
    """Reference enumeration order (plinopt_sparsify.inl:256-268) restated for residues mod p."""
    C = [0, 1, -1]

    def aug(r):
        if r in C:
            return
        inv = pow(r % p, -1, p)
        C.extend([r, -r, inv, (p - inv) % p])
    for row in tm:
        for v in row:
            if v % p:
                aug(int(v))
    i = 2
    while len(C) < c:
        aug(i); i += 1
    return np.array(C[:c], dtype=np.int64)


def time_plan(run, reps):
    st = torch.cuda.current_stream()
    for _ in range(3):
        run(st.cuda_stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        run(st.cuda_stream)
    e1.record(st)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def lincomb_cases(peaks):
    L, _, _ = hm.load_fixture("4x4x4_48_rational")
    for c in (20, 64, 128):
        tms, cfs = [], []
        for blk in range(4):
            TM = [[L[i][4 * blk + t] for i in range(len(L))] for t in range(4)]
            tm = np.array([[(v.numerator % P31) * pow(v.denominator % P31, -1, P31) % P31 for v in row] for row in TM], dtype=np.int64)
            tms.append(tm); cfs.append(coeff_list(tm.tolist(), P31, c))
        plan = capi.LincombPlan(P31, np.stack(tms), 0, np.stack(cfs))
        ms = time_plan(lambda s: plan.run(s), 5 if c >= 64 else 50)
        rl, cl, idx = plan.result()
        cand = plan.candidates
        m = 48
        cpu = {}
        if c == 20:  # the oracle's literal testLinComb loop on the same block-0 problem: 1 core (the reference loop is sequential) and all cores
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
            z = np.zeros((4, 4), dtype=np.int64)
            for nt, key in ((1, "cpu_oracle_candidates_per_s_1core"), (os.cpu_count() or 1, "cpu_oracle_candidates_per_s_allcores")):
                i_hi = 2 if nt == 1 else c
                t0 = time.perf_counter()
                tot = O.lincomb_bench(P31, tms[0], np.ones_like(tms[0]), 0, 0, cfs[0], np.ones_like(cfs[0]), z, np.ones_like(z), 0, i_hi, nthreads=nt)[0]
                cpu[key] = tot / (time.perf_counter() - t0)
            cpu["cpu_threads_all"] = os.cpu_count() or 1
        print(json.dumps({"kernel": "lincomb_kernel<u32,48,modp>", "case": f"4x4x4_48_rational_L, 4 blocks, c={c}", "candidates": cand, **cpu,
                          "ms": ms, "candidates_per_s": cand / ms * 1e3, "compare_add_pairs_per_s": cand * m / ms * 1e3,
                          "ialu_pair_peak": peaks["ialu_pairs_per_s"], "frac_of_ialu_pair_peak": cand * m / ms * 1e3 / peaks["ialu_pairs_per_s"],
                          "best": [int(rl[0]), int(cl[0]), int(idx[0])]}))
        plan.close()


def lincomb_c5_case(peaks):
    """BASELINE C5 shape of the sparsifier search: column blocks of 32x32x32_15096_L (TM = 4 x 15096 per block) mod 2^31-1;
    tiled count + pick kernels (m > 64)."""
    big = hm.load_large_csr(P31)
    if big is None:
        return
    _, r, (L, _, _) = big
    rows, cols, ptr, col, val = L
    nb, c = 16, 20
    TM = np.zeros((nb, 4, rows), dtype=np.int64)
    rowidx = np.repeat(np.arange(rows), np.diff(ptr))
    sel = col < 4 * nb
    TM[col[sel] // 4, col[sel] % 4, rowidx[sel]] = val[sel]
    cfs = np.stack([coeff_list(TM[b].tolist(), P31, c) for b in range(nb)])
    plan = capi.LincombPlan(P31, TM, 0, cfs)
    ms = time_plan(lambda s: plan.run(s), 5)
    rl, cl, idx = plan.result()
    cand = plan.candidates
    print(json.dumps({"kernel": "lincomb_big_count_kernel<u32,modp> + lincomb_big_pick_kernel", "case": f"32x32x32_15096_L, {nb} column blocks (TM 4x15096), c={c}",
                      "candidates": cand, "ms": ms, "candidates_per_s": cand / ms * 1e3, "compare_add_pairs_per_s": cand * rows / ms * 1e3,
                      "frac_of_ialu_pair_peak": cand * rows / ms * 1e3 / peaks["ialu_pairs_per_s"], "best_block0": [int(rl[0]), int(cl[0]), int(idx[0])]}))
    plan.close()


def orbit_cases(peaks):
    """Orbit sweep (src/orbiter.cpp:272-324) on every instantiated shape, both measures; ops per candidate as in SURVEY.md 8d."""
    cases = [("2x2x2_7_Winograd", 28), ("3x3x3_23_58", 24), ("4x4x4_49_156", 22), ("4x4x4_48_rational", 22), ("3x4x7_63_rational", 21)]
    for stem, lg in cases:
        L, R, P = hm.load_fixture(stem)
        mkn = hm.LRP2MM(L, R, P)
        m, k, n = mkn
        r = len(L)
        (Li, dl), (Ri, dr), (Pi, dp) = (hm.scaled(M, np.int32) for M in (L, R, P))
        ops = r * (m * m * k + m * k * k + k * k * n + k * n * n + m * m * n + m * n * n) + r * (m * k + k * n + m * n)
        for measure, name in ((capi.MEASURE_NNZ, "nnz"), (capi.MEASURE_G2, "G2")):
            try:
                plan = capi.OrbitPlan(mkn, Li, Ri, Pi, (dl, dr, dp), measure, capi.MODE_PHILOX, 0x504C494E4F505431)
            except capi.PloError as e:
                print(json.dumps({"kernel": "orbit_sweep_kernel", "case": f"{stem} {name}", "error": str(e)}))
                continue
            B = 1 << lg
            ms = time_plan(lambda s: plan.run(0, B, s), 5)
            best = plan.result()
            print(json.dumps({"kernel": f"orbit_sweep_kernel<{m},{k},{n},philox,{name}>", "case": f"{stem}, 2^{lg} candidates", "ms": ms,
                              "candidates_per_s": B / ms * 1e3, "int32_ops_per_candidate": ops, "int32_ops_per_s": ops * B / ms * 1e3,
                              "frac_of_imad_peak": ops * B / ms * 1e3 / peaks["imad_per_s"], "best": best}))
            if stem in ("2x2x2_7_Winograd", "3x3x3_23_58", "3x4x7_63_rational"):
                # survivor compaction inside the sweep kernel: every candidate at least as good as the winner of a short prefix (well
                # under 1 % of the range survives); timed at the C call, records left in a numpy array
                plan.run(0, 1 << 18, 0)
                thr = plan.result()
                Bs = B
                plan.survivors_array(0, 1 << 16, nnz=thr["nnz"], nno=thr["nno"], score=thr["score"], capacity=1 << 24)  # warm-up
                t0 = time.perf_counter()
                cnt, sv = plan.survivors_array(0, Bs, nnz=thr["nnz"], nno=thr["nno"], score=thr["score"], capacity=1 << 24)
                dt = time.perf_counter() - t0
                print(json.dumps({"kernel": f"{plan.kernel} + survivor compaction in the sweep ({name} threshold) + index sort + gather", "case": f"{stem}, 2^{lg} candidates",
                                  "wall_ms": dt * 1e3, "candidates_per_s": Bs / dt, "survivors": int(cnt), "fraction": cnt / Bs,
                                  "sweep_candidates_per_s": B / ms * 1e3, "vs_sweep_rate": (Bs / dt) / (B / ms * 1e3)}))
            plan.close()


def factor_cases():
    """Factorizer random restarts (plinopt_sparsify.inl:924-990): candidates (row orders) per second; the oracle's exact
    rational backSolver on all host threads beside it.  The first three shapes run factor_sweep_kernel; the shipped 63x62 -ALT
    factor and the factors of the <6,6,6> and <8,8,8> triples run factor_wide_kernel (each line names the kernel of its plan)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    import orbit_any_shape_fixtures as F
    cases = [(f"{stem}_{x}", O.dense_fractions(f"{stem}_{x}"), lg) for stem, x, lg in
             (("4x4x4_48_rational", "L", 22), ("3x4x7_63_rational", "R", 21), ("3x4x7_63_rational", "L", 22), ("3x4x7_63_rational-ALT", "L", 0))]
    cases.append(("Strassen_x_3x3x3_23_58_L", F.kron(O.triple("2x2x2_7_Strassen"), O.triple("3x3x3_23_58"))[0], 0))
    cases.append(("4x4x4_49_156_x_Strassen_L", F.kron(O.triple("4x4x4_49_156"), O.triple("2x2x2_7_Strassen"))[0], 0))
    for name, M, lg in cases:
        r, n = len(M), len(M[0])
        A = np.array([[(v.numerator % P31) * pow(v.denominator % P31, -1, P31) % P31 for v in row] for row in M], dtype=np.uint32)
        plan = capi.FactorPlan(P31, A, n, 0x504C494E4F505431)
        if lg == 0:  # no earlier measurement to match: size the range to about half a second of kernel time
            probe = 1 << 14
            lg = max(14, min(26, int(np.log2(probe * 500.0 / time_plan(lambda s: plan.run(0, probe, s), 1)))))
        B = 1 << lg
        ms = time_plan(lambda s: plan.run(0, B, s), 3)
        best = plan.result()
        kernel = plan.kernel
        plan.close()
        ops = n ** 3 + (r - n) * n * n  # oracle field operations per candidate
        cnt = 4000 if ops < 1e5 else max(64, min(4000, int(2e8 / ops)))
        t0 = time.perf_counter()
        ref = O.factor_sweep(M, n, 0x504C494E4F505431, 0, cnt, table=False)
        cpu = cnt / (time.perf_counter() - t0)
        print(json.dumps({"kernel": kernel, "case": f"{name} ({r}x{n}), k={n}, 2^{lg} row orders", "ms": ms,
                          "candidates_per_s": B / ms * 1e3, "best": best, "cpu_oracle_candidates_per_s": cpu,
                          "cpu_threads": O.lib().orc_num_threads(), "cpu_sample": cnt, "cpu_best_of_sample": ref["best"]}))


def dependency_cases(peaks):
    """dependency Explore (src/dependency.cpp:73-100): combinations tested per second (one compare per coordinate per
    combination), the oracle's literal recursion (1 thread, as the reference) on a smaller level beside it."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    for name, level, c, q in (("4x4x4_48_rational_L", 4, 11, 0), ("4x4x4_48_rational_L", 4, 11, 2147483647), ("3x4x7_63_rational_R", 4, 7, 2147483647),
                              ("3x3x3_23_58_L", 5, 11, 2147483647)):
        M = O.dense_fractions(name)
        capi.depender(M, 2, c, q=q)  # warm-up (context, module load)
        t0 = time.perf_counter()
        got = capi.depender(M, level, c, q=q, max_hits=1 << 18)
        dt = time.perf_counter() - t0
        t0 = time.perf_counter()
        ref = O.depender(M, level - 1, c, p=q)
        cpu_dt = time.perf_counter() - t0
        n = len(M[0])
        print(json.dumps({"kernel": "dependency_kernel", "case": f"{name} level {level} c={len(got['coeffs'])} " + ("over Q (int64)" if q == 0 else f"mod {q}"),
                          "combinations": got["ncand"], "hits": got["nhits"], "wall_s_incl_host": dt, "combinations_per_s": got["ncand"] / dt,
                          "compare_pairs_per_s": got["ncand"] * n / dt, "ialu_pair_peak": peaks["ialu_pairs_per_s"],
                          "cpu_oracle_combinations_per_s": ref["ncand"] / cpu_dt, "cpu_threads": 1, "cpu_sample": f"level {level - 1}: {ref['ncand']} combinations"}))


def mmcheck_case():
    rng = np.random.default_rng(0)
    m = k = n = 32
    r = 15096

    def rand_csr(rows, cols, nnz_row):
        ptr = np.arange(rows + 1, dtype=np.int64) * nnz_row
        col = np.concatenate([np.sort(rng.choice(cols, nnz_row, replace=False)) for _ in range(rows)]).astype(np.int32)
        val = rng.integers(1, P31, rows * nnz_row).astype(np.uint32)
        return (rows, cols, ptr, col, val)
    big = hm.load_large_csr(P31)
    if big is not None:  # the real triple regenerated from the reference's .slp (tools/regen_32x32x32.py)
        _, _, (Lc, Rc, Pc) = big
        name = "32x32x32_15096_{L,R,P} mod 2^31-1"
    else:
        Lc, Rc, Pc = rand_csr(r, 1024, 83), rand_csr(r, 1024, 84), rand_csr(1024, r, 1230)
        name = "synthetic 32x32x32_15096-like CSR"
    nnz = sum(len(c[3]) for c in (Lc, Rc, Pc))
    for B in BATCHES:
        plan = capi.MMcheckPlan(P31, (m, k, n), r, Lc, Rc, Pc, B)
        ms = time_plan(lambda s: plan.run(1, 0, s), 10)
        v, ok = plan.result()
        bytes_csr = nnz * 8
        print(json.dumps({"kernel": "mm_slab_spmm_kernel x3 (Hadamard step fused) + gen + verify", "case": f"{name}, batch={B}",
                          "ms": ms, "samples_per_s": B / ms * 1e3, "modmac_per_s": (nnz + r + m * k * n) * B / ms * 1e3,
                          "csr_stream_GBs_if_read_once": bytes_csr / ms * 1e-6, "verdict": v, "samples_ok": int(ok.sum())}))
        plan.close()


if __name__ == "__main__":
    capi.set_device(0)
    peaks = capi.measure_peaks(5)
    print(json.dumps({"peaks": peaks}))
    if "--orbit-only" in sys.argv:
        orbit_cases(peaks)
        sys.exit(0)
    if "--dep-only" in sys.argv:
        dependency_cases(peaks)
        sys.exit(0)
    if "--factor-only" in sys.argv:
        factor_cases()
        sys.exit(0)
    if "--c5-only" in sys.argv:
        lincomb_c5_case(peaks)
        sys.exit(0)
    if "--mm-only" not in sys.argv:
        lincomb_cases(peaks)
        lincomb_c5_case(peaks)
        orbit_cases(peaks)
        factor_cases()
        dependency_cases(peaks)
    mmcheck_case()
