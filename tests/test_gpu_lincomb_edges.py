"""GPU parity of the sparsifier search at its arithmetic edges, against the CPU oracle (orc_lincomb_search on __int128) and, for whole
pipelines, the Python restatement on fractions (tests/py_sparsifier.py):
  A  moduli between 2^31 and 2^32 (sums of two residues leave 32 bits; the inverse lookup must not apply),
  B  exact integers whose magnitude bound needs 8-byte tables,
  C  T3 staged in several shared-memory tiles (PLO_LINCOMB_TILE_ROWS at small c, the natural tiling at c = 130),
  D  the magnitude guards: the oracle's answer or a clean PLO_E_RANGE / PLO_QUAD_RANGE, never a wrapped one.
Every step compares the exact (rl, cl, index) of lincomb_search, of a batched LincombPlan (and its prefix-range shards) and of
lincomb_quad on both of its paths."""
import itertools
from fractions import Fraction

import numpy as np
import pytest

import oracle_lib as O
import py_sparsifier as PS
from plinopt_b200 import sharding as S
from test_gpu_lincomb import sequential_rows

pytestmark = pytest.mark.gpu

P31 = 2147483647
P_ABOVE = (2147483659, 4294967291)  # the smallest prime above 2^31, the largest below 2^32


# ---- helpers ----------------------------------------------------------------------------------------------------------------------
def exact_rank(rows, p):
    """Rank of integer rows over Q (p == 0) or mod p."""
    R = [[Fraction(int(v)) if p == 0 else int(v) % p for v in r] for r in rows]
    rank, ncol = 0, len(R[0]) if R else 0
    for col in range(ncol):
        piv = next((i for i in range(rank, len(R)) if R[i][col] != 0), None)
        if piv is None:
            continue
        R[rank], R[piv] = R[piv], R[rank]
        inv = 1 / R[rank][col] if p == 0 else pow(R[rank][col], -1, p)
        for i in range(len(R)):
            if i != rank and R[i][col] != 0:
                f = R[i][col] * inv
                R[i] = [a - f * b if p == 0 else (a - f * b) % p for a, b in zip(R[i], R[rank])]
        rank += 1
    return rank


def oracle_step(p, tm, off, num, cf, lcob, init=(-1, -1)):
    rl, cl, idx = O.lincomb_search(p, tm, np.ones_like(tm), off, num, cf, np.ones_like(cf), lcob, np.ones_like(lcob), *init)
    return rl, cl, (None if idx < 0 else idx)


def unkey_rows(res):
    return [(int(a), int(b), None if int(i) == 0xFFFFFFFFFFFFFFFF else int(i)) for a, b, i in zip(*res)]


def check_plan(capi, p, tm, off, cf, prev, init, exp):
    """A batch of two copies of the step, then three prefix-range shards max-merged (plinopt_b200.sharding)."""
    pv = None if prev is None else np.stack([prev, prev])
    plan = capi.LincombPlan(p, np.stack([tm, tm]), off, np.stack([cf, cf]), pv, init[0], init[1])
    try:
        plan.run()
        assert unkey_rows(plan.result()) == [exp, exp]
        c3 = len(cf) ** 3
        parts = []
        for lo, hi in ((0, c3 // 3), (c3 // 3, 2 * c3 // 3 + 1), (2 * c3 // 3 + 1, c3)):
            plan.run_range(lo, hi)
            parts.append(unkey_rows(plan.result())[0])
        assert S.lincomb_unkey(max(S.lincomb_key(*r) for r in parts)) == exp, (parts, exp)
    finally:
        plan.close()


def check_quad(capi, monkeypatch, p, tm, off, cf, prev0, init):
    """The block through lincomb_quad, one-launch and multi-kernel paths: the rows of successive one-row searches."""
    n = tm.shape[0]
    exp = sequential_rows(capi, p, tm, off, cf, prev0, init, None)
    pr = dict(TM=tm, off=off, coeffs=cf, prev_rows=prev0 if off else None, init_rl=init[0], init_cl=init[1])
    for nosmall in (False, True):
        if nosmall:
            monkeypatch.setenv("PLO_QUAD_NOSMALL", "1")
        (status, rows), = capi.lincomb_quad(p, [pr])
        monkeypatch.delenv("PLO_QUAD_NOSMALL", raising=False)
        if not exp and init != (-1, -1):  # the seed kept row 0 and there is no vector to go on with
            assert status == capi.QUAD_SEED and rows == [(init[0], init[1], None)], (nosmall, status, rows)
        else:
            assert rows == exp, (nosmall, rows, exp)
            assert status == (capi.QUAD_DONE if len(rows) == min(4, n - off) else capi.QUAD_MISS)


def walk(capi, monkeypatch, p, tm, cf, seed=(-1, -1), plan=True, quad=True):
    """Every (block, num) step of one localSparsifier call on integer inputs (p == 0: exact integers, else residues): lincomb_search
    equals the oracle; optionally the plan and the quad paths too.  A step without a winner takes the first independent canonical
    vector as its row, as the reference's fallback does.  Returns the number of steps checked."""
    n = tm.shape[0]
    lcob = np.zeros((n, n), dtype=np.int64)
    steps = 0
    for off in range(0, n, 4):
        prev0 = lcob[:off].copy()
        for num in range(min(4, n - off)):
            row = off + num
            init = seed if row == 0 else (-1, -1)
            exp = oracle_step(p, tm, off, num, cf, lcob, init)
            prev = lcob[:row].copy() if row else None
            assert capi.lincomb_search(p, tm, off, cf, prev, *init) == exp, (off, num, exp)
            if plan:
                check_plan(capi, p, tm, off, cf, prev, init, exp)
            steps += 1
            if exp[2] is None:
                for pos in range(n):
                    trial = np.zeros(n, dtype=np.int64); trial[pos] = 1
                    if exact_rank(list(lcob[:row]) + [trial], p) == row + 1:
                        lcob[row] = trial
                        break
                continue
            c = len(cf)
            ids = [exp[2] // c ** 3, (exp[2] // c ** 2) % c, (exp[2] // c) % c, exp[2] % c]
            for t in range(4):
                if off + t < n:
                    lcob[row, off + t] = cf[ids[t]]
        if quad:
            check_quad(capi, monkeypatch, p, tm, off, cf, prev0, seed if off == 0 else (-1, -1))
    return steps


def small_tm(n, m, seed, vals=(0, 0, 0, 1, -1, 1, -1, 2, -2)):
    return np.random.default_rng(seed).choice(vals, size=(n, m)).astype(np.int64)


def modp_inputs(p, n, m, c, seed):
    """A small-integer TM with every column times a random residue in [2^31, p) (zero patterns survive; the entries 1 stay above
    2^31), and a coefficient list 0, 1, -1, 2, -2, then x, -x, 1/x, -1/x for random x in [2^31, p), as residues.  For p < 2^31 the
    same with [p/2, p)."""
    rng = np.random.default_rng(seed)
    lo = 2 ** 31 if p > 2 ** 31 else p // 2  # the upper half of the residues when p < 2^31
    scale = rng.integers(lo, p, size=m)
    tm = np.array([[int(v) * int(s) % p for v, s in zip(row, scale)] for row in small_tm(n, m, seed)], dtype=np.int64)
    cf = [0, 1, p - 1, 2, p - 2]
    while len(cf) < c:
        x = int(rng.integers(lo, p))
        xi = pow(x, -1, p)
        cf += [x, p - x, xi, p - xi]
    return tm, np.array(cf[:c], dtype=np.int64)


def above_2_31(p, n, m, c, seed):
    tm, cf = modp_inputs(p, n, m, c, seed)
    assert (tm >= 2 ** 31).sum() >= m // 4 and (cf >= 2 ** 31).sum() >= 2
    return tm, cf


def wrap_inputs(p, n, m, c, seed):
    """modp_inputs with 8 columns replaced so that w* = (x, 1/x, -x, -1/x) (coefficients 5, 7, 6, 8) vanishes on them through sums of
    residues that leave 32 bits: on columns 0-3 the products a_t = C_t . TM[t] of the first two positions lie in [2^31, p) (the
    one-launch quad kernel adds them), on columns 4-7 the same holds for the products times -TM[3]^-1 (the operands of the inverse
    lookup).  32-bit additions would lose exactly the zeros that make w* the winner (checked by wrapped_misses)."""
    tm, cf = modp_inputs(p, n, m, c, seed)
    rng = np.random.default_rng(seed + 1)
    w = [int(cf[t]) for t in (5, 7, 6, 8)]
    inv = [pow(x, -1, p) for x in w]
    big = lambda: int(rng.integers(2 ** 31, p))  # noqa: E731
    for e in range(8):
        r3 = int(rng.integers(1, p))
        if e < 4:
            a0, a1 = big(), big()
        else:  # operands of the lookup: a_t . (-r3^-1) in [2^31, p)
            a0, a1 = (-big() * r3) % p, (-big() * r3) % p
        a2 = (-(a0 + a1 + w[3] * r3)) % p
        tm[:4, e] = [a0 * inv[0] % p, a1 * inv[1] % p, a2 * inv[2] % p, r3]
    return tm, cf


def wrapped_misses(p, tm, cf, idx, lookup):
    """Zeros of candidate idx that a 32-bit sum (a0 + a1, then + a2, each reduced once) would miss: in the one-launch quad kernel's
    form (lookup False) or in the inverse lookup's, whose operands carry the factor -TM[3]^-1."""
    c, M32 = len(cf), (1 << 32) - 1
    w = [int(cf[(idx // c ** (3 - t)) % c]) for t in range(4)]
    misses = 0
    for e in range(tm.shape[1]):
        a = [w[t] * int(tm[t, e]) % p for t in range(4)]
        if sum(a) % p:
            continue
        if lookup:
            if not tm[3, e]:
                continue
            ni = -pow(int(tm[3, e]), -1, p) % p
            a = [x * ni % p for x in a[:3]] + [w[3]]
        t32 = (a[0] + a[1]) & M32
        t32 -= p if t32 >= p else 0
        t32 = (t32 + a[2]) & M32
        t32 -= p if t32 >= p else 0
        misses += (t32 != a[3]) if lookup else ((p - t32) % p != a[3])
    return misses


# ---- A: moduli between 2^31 and 2^32 ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", P_ABOVE)
@pytest.mark.parametrize("n", [4, 6])
def test_moduli_above_2_31_every_step(capi, monkeypatch, p, n):
    """n = 4 and n = 6 (a partial last block), c = 9, with and without a weight seed that loses or wins.  The first winner's zeros
    need sums that leave 32 bits (the one-launch quad kernel must not take its 32-bit form above 2^31)."""
    tm, cf = wrap_inputs(p, n, 12, 9, seed=n)
    win = oracle_step(p, tm, 0, 0, cf, np.zeros((n, n), dtype=np.int64))[2]
    assert wrapped_misses(p, tm, cf, win, lookup=False) >= 4
    assert walk(capi, monkeypatch, p, tm, cf) == n
    assert walk(capi, monkeypatch, p, tm, cf, seed=(1, 0)) == n
    assert walk(capi, monkeypatch, p, tm, cf, seed=(12, 4), plan=False) == n  # unbeatable: the seed keeps row 0


@pytest.mark.parametrize("p", P_ABOVE)
@pytest.mark.parametrize("m,c", [(65, 5), (200, 7)])
def test_moduli_above_2_31_wide_path(capi, monkeypatch, p, m, c):
    tm, cf = above_2_31(p, 4, m, c, seed=m)
    assert walk(capi, monkeypatch, p, tm, cf, quad=False) == 4


def test_threaded_oracle_equals_literal_oracle():
    """The threaded range search (orc_lincomb_bench over every first coefficient) picks the literal search's winner."""
    for p in (0,) + P_ABOVE:
        tm, cf = modp_inputs(p, 4, 12, 7, seed=3) if p else (small_tm(4, 12, 3), np.array([0, 1, -1, 2, -2, 3, -3], dtype=np.int64))
        z = np.zeros((4, 4), dtype=np.int64)
        lit = oracle_step(p, tm, 0, 0, cf, z)
        _, rl, cl, idx = O.lincomb_bench(p, tm, np.ones_like(tm), 0, 0, cf, np.ones_like(cf), z, np.ones_like(z), 0, len(cf))
        assert (rl, cl, None if idx < 0 else idx) == lit


@pytest.mark.parametrize("p", P_ABOVE)
@pytest.mark.parametrize("c", [33, 40])
def test_moduli_above_2_31_many_coefficients(capi, monkeypatch, p, c):
    """c >= 32 above 2^31: the compare kernels (no inverse lookup: the sum of two residues would not fit 32 bits) give the threaded
    oracle's winner and the same as with PLO_LINCOMB_NOINV=1; the quad multi-kernel path gives the one-row searches' rows."""
    tm, cf = wrap_inputs(p, 4, 16, c, seed=c)
    z = np.zeros((4, 4), dtype=np.int64)
    _, rl, cl, idx = O.lincomb_bench(p, tm, np.ones_like(tm), 0, 0, cf, np.ones_like(cf), z, np.ones_like(z), 0, c)
    assert wrapped_misses(p, tm, cf, idx, lookup=True) >= 4  # an inverse lookup above 2^31 would not find this winner
    got = capi.lincomb_search(p, tm, 0, cf)
    assert got == (rl, cl, None if idx < 0 else idx)
    (status, rows), = capi.lincomb_quad(p, [dict(TM=tm, off=0, coeffs=cf)])
    monkeypatch.setenv("PLO_LINCOMB_NOINV", "1")
    assert capi.lincomb_search(p, tm, 0, cf) == got
    monkeypatch.delenv("PLO_LINCOMB_NOINV")
    assert status == capi.QUAD_DONE and rows == sequential_rows(capi, p, tm, 0, cf, [], (-1, -1), None)


def _same_pipeline(capi, M, q, c):
    CoB, Res, ok, st = capi.sparsifier(M, q, 4, c, True)
    eC, eR, eok, _ = O.sparsifier(M, q, 4, c, True)
    assert ok and eok and st["searches"] > 0
    if q:
        canon = lambda X: [[int(v) % q for v in r] for r in X]  # noqa: E731 (the oracle keeps raw negations, Q3)
        F = PS.Zp(q)
    else:
        canon = lambda X: [[Fraction(v) for v in r] for r in X]  # noqa: E731
        F = PS.QQ()
    assert canon(CoB) == canon(eC) and canon(Res) == canon(eR)
    pC, pR = PS.block_sparsifier(F, M, 4, c, True)
    assert canon(CoB) == canon(pC) and canon(Res) == canon(pR)
    return st


@pytest.mark.parametrize("name", ["4x4x4_48_rational_L", "3x4x7_63_rational_R"])
def test_pipeline_modulo_4294967291(capi, name):
    _same_pipeline(capi, O.dense_fractions(name), 4294967291, 11)


# ---- B: exact integers in 8-byte tables -------------------------------------------------------------------------------------------
CF9 = np.array([0, 1, -1, 2, -2, 3, -3, 4, -4], dtype=np.int64)  # max |C| = 4


def wide_int_tm(n, m, seed, scales):
    """A small-integer TM whose columns are multiplied by the given scales in turn (zero patterns are those of the small TM)."""
    tm = small_tm(n, m, seed)
    return tm * np.array([scales[j % len(scales)] for j in range(m)], dtype=np.int64)


CASES_B = {
    "just_above_2^31": [1, 3, 2 ** 26],                    # 4 . 4 . 2^27 = 2^31
    "near_2^61": [1, 2 ** 56, 5],                         # 4 . 4 . 2^57 = 2^61
    "collide_mod_2^32": [2 ** 32, 2 ** 32 + 1, 1, 2 ** 33 - 1],  # sums that are 0 mod 2^32 but not over Z
}


@pytest.mark.parametrize("case", sorted(CASES_B))
@pytest.mark.parametrize("n", [4, 6])
def test_exact_8_byte_tables_every_step(capi, monkeypatch, case, n):
    tm = wide_int_tm(n, 12, seed=n, scales=CASES_B[case])
    bound = 4 * int(np.abs(CF9).max()) * int(np.abs(tm).max())
    assert 2 ** 31 - 1 <= bound < 2 ** 62
    assert walk(capi, monkeypatch, 0, tm, CF9) == n
    assert walk(capi, monkeypatch, 0, tm, CF9, seed=(2, 1), plan=False) == n


def test_exact_8_byte_tables_collide_only_modulo_2_32(capi, monkeypatch):
    """Columns that are 0 mod 2^32 for every candidate, non-zero over Z for most: a 32-bit table would count them all."""
    tm = np.array([[2 ** 32, 1, 2 ** 32 + 1, 0], [2 ** 32, -1, 1, 2 ** 32], [0, 2, -1, 2 ** 32], [2 ** 33, 0, 0, -2 ** 32]], dtype=np.int64)
    assert walk(capi, monkeypatch, 0, tm, CF9) == 4


@pytest.mark.parametrize("case", sorted(CASES_B))
def test_exact_8_byte_tables_wide_path(capi, monkeypatch, case):
    tm = wide_int_tm(4, 65, seed=65, scales=CASES_B[case])
    assert walk(capi, monkeypatch, 0, tm, CF9[:7], quad=False) == 4


def test_batch_with_one_8_byte_problem(capi):
    """One problem needs 8-byte tables, the others fit 4 bytes: the whole batch runs at width 8 and each problem equals its own
    single call, in a LincombPlan and in lincomb_quad."""
    tms = [small_tm(4, 12, 1), wide_int_tm(4, 12, seed=2, scales=CASES_B["collide_mod_2^32"]), small_tm(4, 12, 3)]
    cfs = [CF9, CF9, CF9[::-1].copy()]
    singles = [capi.lincomb_search(0, tm, 0, cf) for tm, cf in zip(tms, cfs)]
    plan = capi.LincombPlan(0, np.stack(tms), 0, np.stack(cfs))
    plan.run()
    assert unkey_rows(plan.result()) == singles
    plan.close()
    probs = [dict(TM=tm, off=0, coeffs=cf) for tm, cf in zip(tms, cfs)]
    assert capi.lincomb_quad(0, probs) == [capi.lincomb_quad(0, [pr])[0] for pr in probs]


# ---- C: tiled T3 rows -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tile", [1, 3, 4])
@pytest.mark.parametrize("c", [5, 9, 13])
def test_tiled_t3_rows(capi, monkeypatch, tile, c):
    """PLO_LINCOMB_TILE_ROWS cuts T3 into tiles of 1, 3 or 4 rows (not dividing c; smaller than the l range of a thread at c = 13,
    lsplit 4): every step mod p and over Q, with previous rows and a seed, equals the oracle."""
    monkeypatch.setenv("PLO_LINCOMB_TILE_ROWS", str(tile))
    tm, cf = modp_inputs(P31, 6, 16, c, seed=c)
    assert walk(capi, monkeypatch, P31, tm, cf, seed=(1, 0)) == 6
    cfq = np.array([0] + [s * k for k in range(1, c) for s in (1, -1)][:c - 1], dtype=np.int64)
    assert walk(capi, monkeypatch, 0, wide_int_tm(4, 16, seed=c, scales=[1, 2 ** 28]), cfq) == 4


def tiling_130():
    """c = 130 over Q with a maximiser in the second tile: 28 columns on which w* = (7, -11, 13, 65) vanishes (65 is coefficient 129,
    the last row of T3), the other 36 of the small-integer pattern; 8-byte elements, mpad 64."""
    c = 130
    cf = np.array([0] + [s * k for k in range(1, 66) for s in (1, -1)][:c - 1], dtype=np.int64)
    tm = wide_int_tm(4, 64, seed=130, scales=[1, 2 ** 24, 3])
    u = np.random.default_rng(131).integers(-2 ** 18, 2 ** 18, size=(3, 28))
    tm[:3, :28] = 65 * u
    tm[3, :28] = -(7 * u[0] - 11 * u[1] + 13 * u[2])
    wstar = ((13 * c + 22) * c + 25) * c + 129
    assert [int(cf[(wstar // c ** (3 - t)) % c]) for t in range(4)] == [7, -11, 13, 65]
    assert 2 ** 31 <= 4 * 65 * int(np.abs(tm).max()) < 2 ** 62
    return c, cf, tm, wstar


def test_natural_tiling_at_c_130(capi, monkeypatch):
    """8-byte elements, mpad 64, c = 130: 128 T3 rows fit 64 KB, so T3 comes in two tiles (the second of 2 rows), and the maximiser
    lies in the second.  The shard of prefixes with the maximiser's first coefficient equals the threaded oracle over the same range;
    the winner is re-scored exactly on the host, no sampled candidate beats it, and it equals the search with 7-row tiles and the
    plan's; lincomb_quad equals four successive one-row searches."""
    c, cf, tm, wstar = tiling_130()
    i0 = wstar // c ** 3
    z = np.zeros((4, 4), dtype=np.int64)
    _, orl, ocl, oidx = O.lincomb_bench(0, tm, np.ones_like(tm), 0, 0, cf, np.ones_like(cf), z, np.ones_like(z), i0, i0 + 1)
    assert oidx == wstar
    plan = capi.LincombPlan(0, tm, 0, cf)
    plan.run_range(i0 * c * c, (i0 + 1) * c * c)
    assert unkey_rows(plan.result()) == [(orl, ocl, oidx)]
    plan.close()
    rl, cl, idx = got = capi.lincomb_search(0, tm, 0, cf)
    assert (rl, cl, idx) == (orl, ocl, oidx)

    def score(ix):
        w = [int(cf[ix // c ** 3]), int(cf[(ix // c ** 2) % c]), int(cf[(ix // c) % c]), int(cf[ix % c])]
        v = [sum(w[t] * int(tm[t, j]) for t in range(4)) for j in range(tm.shape[1])]
        return sum(x == 0 for x in v), sum(x == 0 for x in w), any(w)
    assert score(idx) == (rl, cl, True)
    rng = np.random.default_rng(130)
    last_tile = [int(q) * c + l for q in rng.integers(0, c ** 3, 300) for l in (128, 129)]  # l in the second tile
    for ix in list(rng.integers(0, c ** 4, 3000)) + last_tile:
        s = score(int(ix))
        assert not s[2] or s[:2] < (rl, cl) or (s[:2] == (rl, cl) and int(ix) >= idx), (ix, s)
    plan = capi.LincombPlan(0, tm, 0, cf)
    plan.run()
    assert unkey_rows(plan.result()) == [got]
    plan.close()
    (status, rows), = capi.lincomb_quad(0, [dict(TM=tm, off=0, coeffs=cf)])
    assert status == capi.QUAD_DONE and rows == sequential_rows(capi, 0, tm, 0, cf, [], (-1, -1), None)
    monkeypatch.setenv("PLO_LINCOMB_TILE_ROWS", "7")
    assert capi.lincomb_search(0, tm, 0, cf) == got
    assert capi.lincomb_quad(0, [dict(TM=tm, off=0, coeffs=cf)]) == [(status, rows)]


# ---- D: guards ---------------------------------------------------------------------------------------------------------------------
def test_exact_width_guard(capi, monkeypatch):
    """4 max|C| max|TM| just below 2^62 is searched exactly (every entry point equals the oracle); at 2^62 every entry point
    returns PLO_E_RANGE."""
    cf = np.array([0, 1, -1, 2, -2, 3, -3], dtype=np.int64)
    tm = small_tm(4, 8, 5)
    tm[:, 0] = [(2 ** 62 - 1) // 12, -1, 1, 0]
    assert 4 * 3 * int(np.abs(tm).max()) < 2 ** 62
    assert walk(capi, monkeypatch, 0, tm, cf) == 4
    tm[0, 0] = 2 ** 60
    cf1 = np.array([0, 1, -1], dtype=np.int64)
    for call in (lambda: capi.lincomb_search(0, tm, 0, cf1), lambda: capi.LincombPlan(0, tm, 0, cf1),
                 lambda: capi.lincomb_quad(0, [dict(TM=tm, off=0, coeffs=cf1)])):
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == capi.E_RANGE


def _device_guard_row(rows, cmax):
    """The row at which quad_prepare's guard trips for winners `rows` (nothing known before the call): the functionals of row 2 are
    the 2x2 minors of w0, w1, those of row 3 the 3x3 minors of w0, w1, w2."""
    lim = (2 ** 62 - 1) // (4 * cmax)
    if len(rows) > 2 and max(abs(rows[0][a] * rows[1][b] - rows[0][b] * rows[1][a]) for a, b in itertools.combinations(range(4), 2)) > lim:
        return 2
    if len(rows) > 3:
        m3 = [abs(round(np.linalg.det(np.array([[float(r[k]) for k in cols] for r in rows[:3]])))) for cols in itertools.combinations(range(4), 3)]
        if max(m3) > lim:
            return 3
    return None


def test_quad_device_guard(capi, monkeypatch):
    """Coefficients 0, +-2^20, +-1 whose winners carry 2^20 in different positions: the 2x2 minors of rows 0 and 1 reach 2^40 > 2^62 /
    (4 . 2^20).  lincomb_quad returns PLO_QUAD_RANGE after the rows it decided, and they equal the oracle's."""
    B = 2 ** 20
    cf = np.array([0, B, -B, 1, -1], dtype=np.int64)
    tm = np.random.default_rng(0).choice([0, 0, 1, -1, B, -B], size=(4, 8)).astype(np.int64)
    lcob = np.zeros((4, 4), dtype=np.int64)
    exp, ws = [], []
    for num in range(4):
        r = oracle_step(0, tm, 0, num, cf, lcob)
        ix = r[2]
        w = [int(cf[ix // 125]), int(cf[(ix // 25) % 5]), int(cf[(ix // 5) % 5]), int(cf[ix % 5])]
        lcob[num] = w
        exp.append(r); ws.append(w)
    t = _device_guard_row(ws, B)
    assert t == 2
    for nosmall in (False, True):
        if nosmall:
            monkeypatch.setenv("PLO_QUAD_NOSMALL", "1")
        (status, rows), = capi.lincomb_quad(0, [dict(TM=tm, off=0, coeffs=cf)])
        assert status == capi.QUAD_RANGE and rows == exp[:t], (nosmall, status, rows, exp)
        # the caller goes on with the one-row entry point, then with lincomb_quad for the remaining row
        assert capi.lincomb_search(0, tm, 0, cf, lcob[:t]) == exp[t]
        (status, rows), = capi.lincomb_quad(0, [dict(TM=tm, off=0, coeffs=cf, prev_rows=lcob[:t + 1])])
        assert status == capi.QUAD_DONE and rows == exp[t + 1:]


def test_functionals_beyond_the_quad_guard(capi):
    """A previous row (1, 2^40, 0, 0) has the annihilator (2^40, -1, 0, 0): with max|C| = 2^20, 4 |phi| max|C| = 2^62 is beyond the
    2^30 of lincomb_quad's filter but within the 2^63 of lincomb_search.  lincomb_search equals the oracle; lincomb_quad sets that
    problem aside with PLO_QUAD_RANGE and no row, and decides the other problems of the call as usual."""
    B = 2 ** 20
    cf = np.array([0, 1, -1, B, -B, 2], dtype=np.int64)
    tm = small_tm(4, 10, 9)
    prev = np.array([[1, 2 ** 40, 0, 0]], dtype=np.int64)
    lcob = np.zeros((4, 4), dtype=np.int64); lcob[0] = prev[0]
    exp = oracle_step(0, tm, 0, 1, cf, lcob)
    assert capi.lincomb_search(0, tm, 0, cf, prev) == exp and exp[2] is not None
    other = dict(TM=small_tm(4, 10, 10), off=0, coeffs=cf[:5].copy())
    got = capi.lincomb_quad(0, [dict(TM=tm, off=0, coeffs=cf, prev_rows=prev), other])
    assert got[0] == (capi.QUAD_RANGE, [])
    assert got[1] == capi.lincomb_quad(0, [other])[0] and got[1][0] == capi.QUAD_DONE


def test_annihilator_times_coefficient_guard(capi):
    """4 |phi| max|C| = 2^63 cannot be evaluated in int64 on the device: PLO_E_RANGE from lincomb_search and the plan."""
    cf = np.array([0, 1, -1, 2 ** 21, -2 ** 21], dtype=np.int64)
    tm = small_tm(4, 10, 9)
    prev = np.array([[1, 2 ** 40, 0, 0]], dtype=np.int64)
    for call in (lambda: capi.lincomb_search(0, tm, 0, cf, prev), lambda: capi.LincombPlan(0, tm, 0, cf, prev)):
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == capi.E_RANGE


# ---- D: the guards inside whole pipeline runs over Q --------------------------------------------------------------------------------
def annihilator_functionals(rows):
    """What the host hands the device for previous rows on 4 positions: the reduced row echelon basis of {phi : phi . w = 0}, each
    functional scaled to integers by its LCD (the basis is unique, so this equals the engine's)."""
    def rref(A):
        A, rk = [r[:] for r in A], 0
        for col in range(4):
            piv = next((i for i in range(rk, len(A)) if A[i][col] != 0), None)
            if piv is None:
                continue
            A[rk], A[piv] = A[piv], A[rk]
            A[rk] = [x / A[rk][col] for x in A[rk]]
            A = [r if i == rk or r[col] == 0 else [a - r[col] * b for a, b in zip(r, A[rk])] for i, r in enumerate(A)]
            rk += 1
        return A[:rk]
    R = rref([[Fraction(int(v)) for v in r] for r in rows])
    pivots = [next(k for k in range(4) if r[k] != 0) for r in R]
    basis = []
    for f in (k for k in range(4) if k not in pivots):
        v = [Fraction(0)] * 4
        v[f] = Fraction(1)
        for r, pc in zip(R, pivots):
            v[pc] = -r[f]
        basis.append(v)
    out = []
    for r in rref(basis):
        lcd = 1
        for x in r:
            lcd = lcd * x.denominator // np.gcd(lcd, x.denominator)
        out.append([int(x * lcd) for x in r])
    return out


def guard_trips(M, c):
    """Runs the pipeline in tests/py_sparsifier.py and, for every localSparsifier call whose rows 0-2 are won by candidates, applies
    lincomb_quad's guards to the integer images the engine would use: the device guard trips at row 2 when a 2x2 minor of rows 0
    and 1 exceeds (2^62 - 1) / (4 max|C|); the host then searches row 2 alone and calls lincomb_quad again with rows 0-2 known, where
    the host guard trips when 4 max|phi| max|C| >= 2^30.  Returns (device trips, host trips after them, largest exact-width bound)."""
    calls = []
    orig, orig_images = PS.local_sparsifier, PS.integer_images

    def local(F, TCoB, TM, maxnumcoeff, trace=None):
        tr = []
        out = orig(F, TCoB, TM, maxnumcoeff, trace=tr)
        calls.append((images[-1], {num: e for _, num, _, _, e, _ in tr}))
        return out
    images = []
    PS.local_sparsifier = local
    PS.integer_images = lambda F, TM, C: images.append(orig_images(F, TM, C)) or images[-1]  # noqa: E731
    try:
        PS.block_sparsifier(PS.QQ(), M, 4, c, True)
    finally:
        PS.local_sparsifier, PS.integer_images = orig, orig_images
    dev = host = 0
    bound = 0
    for (tm, cf), won in calls:
        cf = [int(x) for x in cf]
        cmax, cc = max(abs(x) for x in cf), len(cf)
        bound = max(bound, 4 * cmax * max(abs(int(x)) for x in tm.flat))
        if not all(t in won for t in range(3)):
            continue
        w = [[cf[(won[t] // cc ** (3 - s)) % cc] for s in range(4)] for t in range(3)]
        if max(abs(w[0][a] * w[1][b] - w[0][b] * w[1][a]) for a, b in itertools.combinations(range(4), 2)) > (2 ** 62 - 1) // (4 * cmax):
            dev += 1
            host += 4 * max(abs(x) for r in annihilator_functionals(w) for x in r) * cmax >= 2 ** 30
    return dev, host, bound


def guard_matrix(seed, rows, big):
    vals = [Fraction(0), Fraction(0), Fraction(1), Fraction(-1), Fraction(2), Fraction(3), Fraction(big), Fraction(-big), Fraction(1, big), Fraction(1, 3)]
    rng = np.random.default_rng(seed)
    return [[vals[int(rng.integers(len(vals)))] for _ in range(4)] for _ in range(rows)]


@pytest.mark.parametrize("seed,big", [(106, 4096), (1209, 1024)])
def test_pipeline_through_the_quad_guards(capi, seed, big):
    """Entries 4096 (1024) and their inverses make large integer coefficients whose winners trip lincomb_quad's device guard at row 2;
    the call that follows, with rows 0-2 known, trips the host guard on the functionals (which used to fail the whole run with
    PLO_E_RANGE).  The runs go through the one-row fallback twice, search on 8-byte tables and equal the oracle and the Python
    restatement."""
    M = guard_matrix(seed, 8, big)
    dev, host, bound = guard_trips(M, 7)
    assert dev >= 1 and host >= 1 and 2 ** 31 - 1 <= bound < 2 ** 62
    st = _same_pipeline(capi, M, 0, 7)
    calls = []
    orig = PS.local_sparsifier
    PS.local_sparsifier = lambda *a, **k: calls.append(1) or orig(*a, **k)  # noqa: E731
    try:
        PS.block_sparsifier(PS.QQ(), M, 4, 7, True)
    finally:
        PS.local_sparsifier = orig
    # one lincomb_quad call per localSparsifier call at least, plus one single-row search per guard trip
    assert st["searches"] >= len(calls) + dev + host
