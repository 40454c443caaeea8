"""SLP -> matrix builder (SURVEY.md section 8 row f1: matrixBuilder include/plinopt_programs.inl:1459-1608,
parser :618-686, parenthesisExpand :1615-1679) against the reference's own .slp/.sms pairs
(data/Makefile:31-32 generates one from the other), and the regenerated 32x32x32_15096 triple
(.MISSING_LARGE_BLOBS:1-3) against the matrix-multiplication identity.  Host-only: no GPU needed."""
import json
import os
from fractions import Fraction

import numpy as np
import pytest

from plinopt_b200 import capi, hm

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PROGRAMS = json.load(open(os.path.join(GOLD, "slp_programs.json")))
MATRICES = json.load(open(os.path.join(GOLD, "hm_matrices.json")))


def _entries(rows, ptr, col, num, den):
    return {(i, int(col[t])): Fraction(int(num[t]), int(den[t])) for i in range(rows) for t in range(ptr[i], ptr[i + 1])}


@pytest.mark.parametrize("name", sorted(PROGRAMS))
def test_program_rebuilds_the_shipped_matrix(name):
    rows, cols, ptr, col, num, den = capi.slp_to_csr(PROGRAMS[name])
    M = MATRICES[name]
    assert (rows, cols) == (M["rows"], M["cols"])
    assert _entries(rows, ptr, col, num, den) == {(i, j): Fraction(v) for i, j, v in M["entries"]}
    assert all(ptr[i] == ptr[i + 1] or np.all(np.diff(col[ptr[i]:ptr[i + 1]]) > 0) for i in range(rows))  # sorted columns


def test_syntax_forms():
    """Line forms seen in data/: sums, parentheses with a rational factor, reuse of an output on its own
    right-hand side, comments, several statements per line, cancellation to zero."""
    text = "# comment\nt1:=i0+i1; t2:=(i2-i0)*15/17-i1*2/17+t1;\no0:=t2;\no1:=i3;\no1:=o1-i3+i0/4;\no2:=-(i1+i2)*3;\n"
    rows, cols, ptr, col, num, den = capi.slp_to_csr(text)
    assert (rows, cols) == (3, 4)
    e = _entries(rows, ptr, col, num, den)
    assert e == {(0, 0): Fraction(2, 17), (0, 1): Fraction(15, 17), (0, 2): Fraction(15, 17), (1, 0): Fraction(1, 4),
                 (2, 1): Fraction(-3), (2, 2): Fraction(-3)}


@pytest.mark.parametrize("bad", ["o0:=i0+;", "o0:=(i0;", "o0 i1;", "o0:=i0*x;", "o0:=i0/0;", "o0:=3+i0;"])
def test_parse_errors_are_reported_not_fatal(bad):
    with pytest.raises(capi.PloError):
        capi.slp_to_csr(bad)


def _spmv(shape, ptr, col, val, x, p):
    y = np.zeros(shape[0], dtype=np.int64)
    prod = (val.astype(np.int64) * x[col]) % p  # p < 2^20: products < 2^40, row sums of < 2^14 terms stay < 2^63
    np.add.at(y, np.repeat(np.arange(shape[0]), np.diff(ptr)), prod)
    return y % p


def test_regenerated_32x32x32_is_a_matrix_multiplication_algorithm():
    """SURVEY.md section 0.6: 15096x1024 / 15096x1024 / 1024x15096 with 1257376 / 1260960 / 1259424 non-zeroes;
    P((L a) o (R b)) = vec(A B) (plinopt_library.inl:472-558), here in numpy mod 1000003."""
    big = hm.load_large_csr(1000003)
    assert big is not None, "tests/golden/large/32x32x32_15096.npz missing: run tools/regen_32x32x32.py"
    (m, k, n), r, (L, R, P) = big
    assert [(c[0], c[1], len(c[3])) for c in (L, R, P)] == [(15096, 1024, 1257376), (15096, 1024, 1260960), (1024, 15096, 1259424)]
    p = 1000003
    rng = np.random.default_rng(3)
    A = rng.integers(0, p, (m, k)); B = rng.integers(0, p, (k, n))
    h = (_spmv(L[:2], L[2], L[3], L[4], A.reshape(-1), p) * _spmv(R[:2], R[2], R[3], R[4], B.reshape(-1), p)) % p
    c = _spmv(P[:2], P[2], P[3], P[4], h, p)
    Cm = np.array([[sum(int(A[i, t]) * int(B[t, j]) for t in range(k)) % p for j in range(n)] for i in range(m)])
    assert np.array_equal(c, Cm.reshape(-1))


def test_large_fixture_decodes_to_the_regenerated_csr(tmp_path):
    """hm.load_large returns exactly the CSR arrays tools/regen_32x32x32.py produced (digest of their dtypes, shapes and bytes,
    taken from the plain-CSR file it wrote before the compact encoding), and hm.save_large re-encodes them losslessly."""
    import hashlib
    z = hm.load_large()
    assert z is not None
    h = hashlib.sha256()
    for x in "LRP":
        for f in ("shape", "ptr", "col", "num", "den"):
            a = z[f"{x}_{f}"]
            h.update(f"{x}_{f}:{a.dtype.str}:{a.shape}".encode())
            h.update(np.ascontiguousarray(a).tobytes())
    assert h.hexdigest() == "8550a46ac88fc52e513170dee9bf7d2c91b953da2a4981bab855c7b67df2d8cc"
    hm.save_large(str(tmp_path / "again.npz"), z)
    again = hm.load_large(str(tmp_path / "again.npz"))
    assert sorted(again) == sorted(z)
    for key in z:
        assert again[key].dtype == z[key].dtype and np.array_equal(again[key], z[key]), key
