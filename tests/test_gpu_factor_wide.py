"""GPU parity of the Factorizer search beyond factor_sweep_kernel's reach: up to 64 columns and 512 rows (factor_wide_kernel).
The shipped tall -ALT factors (48x47, 63x62) and the factors of the <6,6,6> to <8,8,8> triples the orbit sweep runs, candidate by
candidate against the oracle's restatement of backSolver (include/plinopt_sparsify.inl:755-867, 924-990), then the driver and the
CLI on the same inputs."""
import functools
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import orbit_any_shape_fixtures as F
from plinopt_b200 import hm
from test_orbit_large_host import fixtures as large_triples

pytestmark = pytest.mark.gpu
P31 = 2147483647
SEED = 0x504C494E4F505431
BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin")

ALT = [f"{stem}-ALT_{x}" for stem in ("4x4x4_48_rational", "4x4x4_48_accurate", "3x4x7_63_rational") for x in "LR"]


def residues(M, p):
    return np.array([[(v.numerator % p) * pow(v.denominator % p, -1, p) % p for v in row] for row in M], dtype=np.uint32)


def tall(M):
    return [list(c) for c in zip(*M)] if len(M) < len(M[0]) else [list(row) for row in M]


@functools.lru_cache(maxsize=None)
def large():
    """Factors of the triples beyond the orbit sweep's constant bank, P in its tall orientation P^T."""
    T = large_triples()
    s = T["Strassen_x_3x3x3_23_58"]
    return {"Strassen_x_3x3x3_23_58_L": s[0], "Strassen_x_3x3x3_23_58_R": s[1], "Strassen_x_3x3x3_23_58_PT": tall(s[2]),
            "naive_7x7x7_L": T["naive_7x7x7"][0], "4x4x4_49_156_x_Strassen_L": T["4x4x4_49_156_x_Strassen"][0],
            "naive_8x8x8_L": F.naive(8, 8, 8)[0]}


def matrix(name):
    return [list(row) for row in O.dense_fractions(name)] if name in ALT else large()[name]


def rate_count(r, n, k):
    """A candidate range the oracle sweeps in seconds: one candidate costs it about n^3 + (r - k) n^2 field operations."""
    ops = n ** 3 + (r - k) * n * n
    return max(64, min(600, int(4e9 / ops))), max(16, min(200, int(4e8 / ops)))


CASES = [(a, "n") for a in ALT] + [(a, "r") for a in ALT] + [(m, "n") for m in ("Strassen_x_3x3x3_23_58_L", "Strassen_x_3x3x3_23_58_R",
                                                                                 "Strassen_x_3x3x3_23_58_PT", "naive_7x7x7_L",
                                                                                 "4x4x4_49_156_x_Strassen_L", "naive_8x8x8_L")]


@pytest.mark.parametrize("name,kk", CASES)
def test_candidate_table_matches_oracle(capi, name, kk):
    M = matrix(name)
    r, n = len(M), len(M[0])
    k = n if kk == "n" else r
    assert n > 32 or r > 255
    A = residues(M, P31)
    plan = capi.FactorPlan(P31, A, k, SEED)
    assert plan.kernel.startswith("factor_wide_kernel<%d>" % (2 if n > 32 else 1))
    plan.close()
    cnt, exact_cnt = rate_count(r, n, k)
    best, tab = capi.factor_sweep(P31, A, k, SEED, 10, 10 + cnt, table=True)
    ref = O.factor_sweep(M, k, SEED, 10, 10 + cnt, p=P31)
    assert np.array_equal(tab, ref["table"])
    assert best == ref["best"]
    # the exact rational oracle on a shorter range: scoring modulo a 31-bit prime sees the same zero / +-1 pattern
    exact = O.factor_sweep(M, k, SEED, 10, 10 + exact_cnt)
    assert np.array_equal(tab[:exact_cnt], exact["table"])


def random_matrix(rng, r, n, p, deficient=False):
    """Sparse-ish residues: zeros, +-1 and arbitrary values, so that every part of the score is exercised."""
    kind = rng.integers(0, 4, size=(r, n))
    vals = rng.integers(1, p, size=(r, n), dtype=np.int64)
    A = np.where(kind == 0, 0, np.where(kind == 1, 1, np.where(kind == 2, p - 1, vals))).astype(np.int64)
    if deficient:  # last column = twice the first: rank below n
        A[:, n - 1] = (2 * A[:, 0]) % p
    return A.astype(np.uint32)


RANDOM = [(33, 33), (40, 100), (47, 211), (48, 48), (63, 300), (64, 64), (64, 512), (1, 256), (5, 300), (17, 400), (32, 512), (32, 256)]


@pytest.mark.parametrize("p", [3, 101, P31])
@pytest.mark.parametrize("n,r", RANDOM)
def test_factor_sweep_random_matrices(capi, n, r, p):
    rng = np.random.default_rng(n * 1000 + r + p % 1000)
    A = random_matrix(rng, r, n, p)
    M = [[O.Fraction(int(v)) for v in row] for row in A]
    for k in sorted({n, int(rng.integers(n, r + 1)), r}):
        cnt = max(8, min(96, rate_count(r, n, k)[0] // 2))
        best, tab = capi.factor_sweep(p, A, k, SEED, 3, 3 + cnt, table=True)
        ref = O.factor_sweep(M, k, SEED, 3, 3 + cnt, p=p)
        assert np.array_equal(tab, ref["table"]), (n, r, k, p)
        assert best == ref["best"], (n, r, k, p)


@pytest.mark.parametrize("n,r", [(2, 300), (40, 90), (64, 512)])
def test_rank_deficient_inputs_have_no_winner(capi, n, r):
    rng = np.random.default_rng(n + r)
    A = random_matrix(rng, r, n, 101, deficient=True)
    best, tab = capi.factor_sweep(101, A, n, SEED, 0, 64, table=True)
    assert best[3] is None
    assert (tab[:, 0] == 0xFFFFFFFF).all() and (tab[:, 1:] == 0).all()


def test_row_order_decode_is_the_oracles(capi):
    for r in (256, 343, 512):
        for idx in (0, 1, 12345, 2**40 + 17):
            got = capi.factor_decode(r, SEED, idx)
            assert got.tolist() == O.factor_decode(r, SEED, idx).tolist()
            assert sorted(got.tolist()) == list(range(r))


def test_large_sweep_winner_is_reproducible_and_exact(capi):
    """Any split of a 2^20-candidate range gives the same winner; the winner's score is the exact oracle's for that candidate
    and Alt . CoB == M holds exactly."""
    M = matrix("4x4x4_48_rational-ALT_L")
    n = len(M[0])
    A = residues(M, P31)
    N = 1 << 20
    whole = capi.factor_sweep(P31, A, n, SEED, 0, N)
    for cut in (N // 3, 12345, N - 1):
        halves = [capi.factor_sweep(P31, A, n, SEED, 0, cut), capi.factor_sweep(P31, A, n, SEED, cut, N)]
        assert whole == min(halves, key=lambda b: (b[0], b[1], b[2], b[3]))
    exact = O.factor_sweep(M, n, SEED, whole[3], whole[3] + 1, matrices=True)
    assert tuple(int(v) for v in exact["table"][0]) == whole[:3]
    prod = [[sum(exact["alt"][i][t] * exact["cob"][t][j] for t in range(n)) for j in range(n)] for i in range(len(M))]
    assert prod == M
    first = O.factor_sweep(M, n, SEED, 0, 2000)["best"]
    assert whole[:3] <= first[:3]


@pytest.mark.parametrize("ndev", [2, 8])
def test_sweep_devices_equals_single_device(capi, ndev):
    """plo_factor_sweep_devices shards the range over ndev devices through the plan; the winner is the single-device one."""
    if capi.device_count() < ndev:
        pytest.skip(f"needs {ndev} devices")
    for name in ("3x4x7_63_rational-ALT_L", "naive_8x8x8_L"):
        M = matrix(name)
        n = len(M[0])
        A = residues(M, P31)
        N = 1 << 14
        assert capi.factor_sweep_devices(ndev, P31, A, n, SEED, 0, N) == capi.factor_sweep(P31, A, n, SEED, 0, N)


@pytest.mark.parametrize("name,r,n", [("4x4x4_48_rational_L", 48, 16), ("3x4x7_63_rational_R", 63, 28), ("3x4x7_63_rational_L", 63, 12)])
def test_shapes_within_the_first_kernel_keep_it(capi, name, r, n):
    """n <= 32 and r <= 255 stay on factor_sweep_kernel<N> (N = n rounded up to a multiple of 4), whatever the inner dimension."""
    A = residues(O.dense_fractions(name), P31)
    assert A.shape == (r, n)
    for k in (n, r):
        plan = capi.FactorPlan(P31, A, k, SEED)
        assert plan.kernel == "factor_sweep_kernel<%d>" % ((n + 3) // 4 * 4)
        plan.close()
    rng = np.random.default_rng(7)
    for r2, n2 in ((255, 32), (256, 32), (100, 33)):
        plan = capi.FactorPlan(101, random_matrix(rng, r2, n2, 101), n2, SEED)
        assert plan.kernel == ("factor_sweep_kernel<32>" if r2 <= 255 and n2 <= 32 else "factor_wide_kernel<%d>" % (1 if n2 <= 32 else 2))
        plan.close()


@pytest.mark.parametrize("name,q", [(a, q) for a in ALT for q in (0, 7)] + [(m, 0) for m in ("Strassen_x_3x3x3_23_58_L", "Strassen_x_3x3x3_23_58_R",
                                                                                             "Strassen_x_3x3x3_23_58_PT", "naive_7x7x7_L",
                                                                                             "4x4x4_49_156_x_Strassen_L", "naive_8x8x8_L")])
def test_factorizer_driver(capi, name, q):
    """plo_factorizer: a consistent factorisation never worse than M = M.I (:958), with the same winner, Alt and CoB as the
    oracle's exact sweep over the same candidates."""
    M = matrix(name)
    r, n = len(M), len(M[0])
    loops = 64
    rc, Alt, CoB, rep = capi.factorizer(M, q=q, loops=loops, seed=5)
    assert rc == 0 and rep["consistent"] and rep["final"] <= rep["initial"]
    ref = O.factor_sweep(M, n, 5, 0, loops, p=q, matrices=True)
    if ref["best"][:3] < rep["initial"]:
        assert rep["index"] == ref["best"][3] and rep["final"] == ref["best"][:3]
        assert Alt == ref["alt"] and CoB == ref["cob"]
    else:
        assert rep["index"] is None and rep["final"] == rep["initial"]
    if q == 0:
        assert [[sum(Alt[i][t] * CoB[t][j] for t in range(n)) for j in range(n)] for i in range(r)] == M


def test_limits(capi):
    """Beyond 64 columns or 512 rows: the error class 33 columns got before the wide kernel existed (PLO_E_ARG from the sweep,
    PLO_E_SHAPE from the driver), with the limit in the message."""
    rng = np.random.default_rng(1)
    for r, n in ((100, 65), (513, 8), (513, 64)):
        A = random_matrix(rng, r, n, 101)
        with pytest.raises(capi.PloError) as e:
            capi.factor_sweep(101, A, n, SEED, 0, 8)
        assert e.value.code == capi.E_ARG and "n <= 64" in str(e.value) and "512" in str(e.value)
    A = random_matrix(rng, 512, 64, 101)
    assert capi.factor_sweep(101, A, 64, SEED, 0, 8)[3] is not None
    M = [[O.Fraction(int(v)) for v in row] for row in random_matrix(rng, 100, 65, 101)]
    with pytest.raises(capi.PloError) as e:
        capi.factorizer(M, loops=2)
    assert e.value.code == capi.E_SHAPE and "64 columns" in str(e.value)


def test_factorizer_cli(capi, tmp_path):
    """`factorizer -O 10` and `factorizer -q 7` (bin/FDT.sh:69-76) on a shipped 63x62 factor; a wide matrix gets the reference's
    inner-dimension failure."""
    exe = os.path.join(BIN, "factorizer")
    f = tmp_path / "3x4x7_63_rational-ALT_L.sms"
    hm.write_sms(O.dense_fractions("3x4x7_63_rational-ALT_L"), str(f))
    for flags in (["-O", "10"], ["-q", "7"]):
        p = subprocess.run([exe] + flags + [str(f)], capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr
        assert "SUCCESS: consistent factorization!" in p.stderr and "63x62 by 62x62" in p.stderr
    w = tmp_path / "4x4x4_48_rational_P.sms"
    hm.write_sms(O.dense_fractions("4x4x4_48_rational_P"), str(w))
    p = subprocess.run([exe, "-O", "10", str(w)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 255 and "Fail: inner dimension has to be between 48 and 16." in p.stderr
