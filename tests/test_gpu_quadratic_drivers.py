"""GPU tests of the `-P "X^2-d"` drivers: plo_mmchecker_quad (exact over Q(sqrt d) at the sampled points, two embeddings per split
prime), plo_orbiter_quad / plo_orbiter_progress_quad against plans and the oracle's exact transform applied to each part, and the
CLIs bin/MMchecker, bin/orbiter and bin/growthfactor with `-P`."""
import os
import subprocess

import pytest

import oracle_lib as O
from plinopt_b200 import hm
from test_quadratic_host import FX, G2_DPS_ACCURATE, dps_accurate, is_algorithm_quad, rational, scaled_quad

pytestmark = pytest.mark.gpu
BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin")
SEED = 0x504C494E4F505431  # the CLIs' default seed


def count_quad(T):
    """(nnz, nno) over Q(sqrt d): zero iff both parts are zero, +-1 iff the sqrt(d) part is zero and the rational part is +-1."""
    nnz = nno = 0
    for A, B in T:
        for ra, rb in zip(A, B):
            for a, b in zip(ra, rb):
                if a != 0 or b != 0:
                    nnz += 1
                    nno += not (b == 0 and abs(a) == 1)
    return nnz, nno


def is_prime(x):
    if x < 2:
        return False
    for q in (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37):
        if x % q == 0:
            return x == q
    s, t = 0, x - 1
    while t % 2 == 0:
        s, t = s + 1, t // 2
    for a in (2, 3, 5, 7, 11, 13, 17):
        y = pow(a, t, x)
        if y in (1, x - 1):
            continue
        for _ in range(s - 1):
            y = y * y % x
            if y == x - 1:
                break
        else:
            return False
    return True


def first_split_prime(d, dens):
    """The first prime of the check from 2^31 - 1 downwards: d a non-zero square, no denominator vanishing."""
    p = 2 ** 31 - 1
    while not (is_prime(p) and d % p and pow(d % p, (p - 1) // 2, p) == 1 and all(x % p for x in dens)):
        p -= 2
    return p


def sqrt_mod(a, p):
    """Tonelli-Shanks: a square root of a modulo the odd prime p."""
    a %= p
    q, s = p - 1, 0
    while q % 2 == 0:
        q, s = q // 2, s + 1
    z = 2
    while pow(z, (p - 1) // 2, p) != p - 1:
        z += 1
    m, c, t, r = s, pow(z, q, p), pow(a, q, p), pow(a, (q + 1) // 2, p)
    while t != 1:
        i, u = 0, t
        while u != 1:
            u, i = u * u % p, i + 1
        b = pow(c, 1 << (m - i - 1), p)
        m, c, t, r = i, b * b % p, t * b * b % p, r * b % p
    return r


def denominators(T):
    return {v.denominator for A, B in T for M in (A, B) for row in M for v in row}


def with_p_entry(T, da, db, e=0, l=0):
    """T with P[e][l] += da + db.sqrt(d)."""
    (L, R, (Pa, Pb)) = T
    Pa, Pb = [list(r) for r in Pa], [list(r) for r in Pb]
    Pa[e][l] += da
    Pb[e][l] += db
    return L, R, (Pa, Pb)


# ---------------------------------------------------------------- MMchecker over Q(sqrt d)
@pytest.mark.parametrize("name", sorted(FX))
def test_mmchecker_accepts_every_fixture(capi, name):
    d, T = FX[name]
    v, cnt, npr = capi.mmchecker_quad(d, *T)
    assert v == 0 and npr >= 1
    assert cnt == count_quad(T)


def test_mmchecker_refuses_what_is_not_an_algorithm(capi):
    (La, Lb), R, P = dps_accurate()
    Lb = [list(row) for row in Lb]
    i, j = next((i, j) for i, row in enumerate(Lb) for j, v in enumerate(row) if v != 0)
    Lb[i][j] = -Lb[i][j]  # the conjugated entry of test_a_wrong_sign_of_sqrt_d_is_not_an_algorithm
    assert capi.mmchecker_quad(3, (La, Lb), R, P)[0] == 1
    assert capi.mmchecker_quad(2, *dps_accurate())[0] == 1  # DPS-accurate read over Q(sqrt 2)


@pytest.mark.parametrize("stem", ["2x2x2_7_Strassen", "2x2x2_7_DPS-accurate", "3x3x3_23_58"])
def test_zero_sqrt_d_parts_give_the_rational_verdict(capi, stem):
    T = O.triple(stem)
    assert capi.mmchecker_quad(3, *rational(T))[0] == capi.mmchecker_bits(*T)[0]


def test_mmchecker_is_exact_beyond_the_first_prime(capi):
    """An error divisible by the first split prime p1 passes modulo p1 under both embeddings; the next prime must catch it."""
    T = dps_accurate()
    p1 = first_split_prime(3, denominators(T))
    v, _, npr = capi.mmchecker_quad(3, *with_p_entry(T, p1, 0))
    assert v == 1 and npr >= 2


@pytest.mark.parametrize("root_index", [0, 1])
def test_mmchecker_uses_both_embeddings(capi, root_index):
    """The error -r + sqrt(d), r^2 = d mod p1, vanishes under one embedding of p1 only: the other one must catch it at p1."""
    T = dps_accurate()
    p1 = first_split_prime(3, denominators(T))
    r = sqrt_mod(3, p1)
    r = (r, p1 - r)[root_index]
    v, _, npr = capi.mmchecker_quad(3, *with_p_entry(T, -r, 1))
    assert v == 1 and npr == 1


# ---------------------------------------------------------------- Orbiter over Q(sqrt d)
CASES = [("DPS-accurate", 0, 48 ** 3), ("2x2x2_7_Winograd_sqrt2", 1, 20000), ("DPS-accurate_kron_Strassen", 1, 2000)]


def apply_parts(T, U, V, W):
    """The oracle's exact transform applied to the rational and to the sqrt(d) part."""
    A = O.orbit_apply(*(M[0] for M in T), U, V, W)
    B = O.orbit_apply(*(M[1] for M in T), U, V, W)
    return tuple(zip(A, B))


def same(X, Y):
    return all([list(r) for r in Xp] == [list(r) for r in Yp] for x, y in zip(X, Y) for Xp, Yp in zip(x, y))


@pytest.mark.parametrize("name,mode,loops", CASES)
@pytest.mark.parametrize("measure", [0, 3])
def test_orbiter_quad(capi, name, mode, loops, measure):
    d, T = FX[name]
    Lj, Rg, hP, rep = capi.orbiter_quad(d, *T, measure=measure, mode=mode, seed=77, loops=loops)
    mkn, parts, dens = scaled_quad(T)
    plan = capi.OrbitPlan.quad(d, mkn, *parts, dens, measure, mode, 77)
    plan.run(0, loops)
    best = plan.result()
    plan.close()
    assert rep["best"] == best
    out = (Lj, Rg, hP)
    assert rep["mm_verdict"] == 0 and is_algorithm_quad(out, d)
    init = count_quad(T)
    assert (rep["init_nnz"], rep["init_nno"]) == init
    if measure == 3:
        assert abs(rep["init_score"] - capi.growth_factors_quad(d, *T)["G2"]) <= 1e-12 * rep["init_score"]
    if rep["improved"]:
        U, V, W = capi.orbit_decode(*mkn, mode, 77, best["index"])
        assert same(out, apply_parts(T, U, V, W))
        if measure == 3:
            assert best["score"] < rep["init_score"] * (1 - 1e-12)
            assert abs(best["score"] - capi.growth_factors_quad(d, *out)["G2"]) <= 1e-12 * best["score"]
        else:
            assert (best["nnz"], best["nno"]) < init and (best["nnz"], best["nno"]) == count_quad(out)
    else:
        assert same(out, T)
    recs = capi.orbiter_progress_quad(d, *T, measure=measure, mode=mode, seed=77, loops=loops)
    assert bool(recs) == rep["improved"]
    key = (lambda b: b["score"]) if measure == 3 else (lambda b: (b["nnz"], b["nno"]))
    for a, b in zip(recs, recs[1:]):
        assert a["index"] < b["index"] and key(b) < key(a)
    if recs:
        assert recs[-1] == rep["best"]


def test_orbiter_quad_over_two_devices(capi):
    if capi.device_count() < 2:
        pytest.skip("needs two devices")
    d, T = FX["DPS-accurate_kron_Strassen"]
    try:
        one = capi.orbiter_quad(d, *T, measure=3, seed=5, loops=3000)
        capi.lib().plo_set_sweep_devices(2)
        two = capi.orbiter_quad(d, *T, measure=3, seed=5, loops=3000)
    finally:
        capi.lib().plo_set_sweep_devices(1)
    assert one == two


# ---------------------------------------------------------------- CLIs
def write_quad(tmp_path, stem, T):
    paths = []
    for x, M in zip("LRP", T):
        p = tmp_path / f"{stem}_{x}.sms"
        hm.write_sms_quad(M, str(p))
        paths.append(str(p))
    return paths


def run(exe, args):
    return subprocess.run([os.path.join(BIN, exe)] + args, capture_output=True, text=True, timeout=600)


def test_mmchecker_cli_dps_accurate_x(capi, tmp_path):
    """The fourth mmcheck line of the reference's Makefile: `MMchecker -P "X^2-3"` on 2x2x2_7_DPS-accurate-X."""
    files = write_quad(tmp_path, "2x2x2_7_DPS-accurate-X", dps_accurate())
    p = run("MMchecker", ["-P", "X^2-3"] + files)
    assert p.returncode == 0 and "SUCCESS: correct 2x2x2" in p.stderr, p.stderr
    assert "# over Q(sqrt 3): 32 points of 32-bit coordinates, decided modulo" in p.stderr and "two embeddings each" in p.stderr
    p = run("MMchecker", ["-P", "X^2-2"] + files)
    assert p.returncode == 1 and "not a 2x2x2 MM algorithm" in p.stderr


def test_orbiter_cli_writes_x_files(capi, tmp_path):
    d, T = FX["2x2x2_7_Winograd_sqrt2"]
    files = write_quad(tmp_path, "winograd_sqrt2", T)
    loops = 48 ** 3
    p = run("orbiter", ["-P", "X^2-2", "-g", "--exhaustive", "-O", str(loops)] + files)
    assert p.returncode == 0, p.stderr
    assert "SUCCESS: correct 2x2x2" in p.stderr and "# Found opt:" in p.stderr and "Rdcd. opt" in p.stderr
    outs = [f.replace(".sms", ".nnz.sms") for f in files]
    got = tuple(hm.read_sms_quad(o) for o in outs)
    Lj, Rg, hP, rep = capi.orbiter_quad(d, *T, measure=3, mode=0, seed=SEED, loops=loops)
    assert rep["improved"] and same(got, (Lj, Rg, hP))
    assert capi.growth_factors_quad(d, *got)["G2"] < 15.0  # Winograd's 17.85 -> a Strassen-like 14.83 point
    q = run("MMchecker", ["-P", "X^2-2"] + outs)
    assert q.returncode == 0 and "SUCCESS: correct 2x2x2" in q.stderr


def test_growthfactor_cli(capi, tmp_path):
    files = write_quad(tmp_path, "dps", dps_accurate())
    p = run("growthfactor", ["-P", "X^2-3"] + files)
    assert p.returncode == 0, p.stderr
    assert "## G2:\t\t12.066031\t" in p.stderr
    assert abs(capi.growth_factors_quad(3, *dps_accurate())["G2"] - G2_DPS_ACCURATE) <= 1e-12 * G2_DPS_ACCURATE
