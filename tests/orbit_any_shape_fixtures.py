"""Algorithms of shapes without a compiled orbit kernel, built from the shipped ones: naive <m,k,n>, Kronecker products (numpy
kron of the row-reshaped factors) and the two rotations of 3x4x7_63_rational.  Triples are lists of rows of Fraction, as
oracle_lib.triple returns them."""
from fractions import Fraction

import numpy as np

import oracle_lib as O


def naive(m, k, n):
    """The schoolbook algorithm: one product a[i][j] b[j][l] per (i, j, l), added to c[i][l]."""
    r = m * k * n
    L = [[Fraction(0)] * (m * k) for _ in range(r)]
    R = [[Fraction(0)] * (k * n) for _ in range(r)]
    P = [[Fraction(0)] * r for _ in range(m * n)]
    t = 0
    for i in range(m):
        for j in range(k):
            for l in range(n):
                L[t][i * k + j] = Fraction(1)
                R[t][j * n + l] = Fraction(1)
                P[i * n + l][t] = Fraction(1)
                t += 1
    return L, R, P


def _obj(M):
    return np.array([[Fraction(v) for v in row] for row in M], dtype=object)


def kron(A, B):
    """<m1 m2, k1 k2, n1 n2> of rank r1 r2 from <m1,k1,n1> (x) <m2,k2,n2>: row t of L (of R) is the Kronecker product of the
    reshaped rows, column t of P that of the reshaped columns."""
    (LA, RA, PA), (LB, RB, PB) = A, B
    (m1, k1, n1), (m2, k2, n2) = O.LRP2MM(*A), O.LRP2MM(*B)
    LA, RA, PA, LB, RB, PB = map(_obj, (LA, RA, PA, LB, RB, PB))
    rA, rB = LA.shape[0], LB.shape[0]
    L, R, Pt = [], [], []
    for a in range(rA):
        for b in range(rB):
            L.append(np.kron(LA[a].reshape(m1, k1), LB[b].reshape(m2, k2)).reshape(-1))
            R.append(np.kron(RA[a].reshape(k1, n1), RB[b].reshape(k2, n2)).reshape(-1))
            Pt.append(np.kron(PA[:, a].reshape(m1, n1), PB[:, b].reshape(m2, n2)).reshape(-1))
    P = np.array(Pt, dtype=object).T
    return [list(x) for x in L], [list(x) for x in R], [list(x) for x in P]


def rotations(stem):
    """The left and right rotations (bin/rotater) of a shipped algorithm, through the oracle."""
    T = O.triple(stem)
    return O.rotater(*T), O.rotater(*T, right=True)


def fixtures():
    """name -> triple.  Every shape here has no compiled orbit kernel."""
    out = {}
    left, right = rotations("3x4x7_63_rational")
    for T in (left, right):
        m, k, n = O.LRP2MM(*T)
        out[f"{m}x{k}x{n}_63_rotated"] = T
    for stem in ("2x2x2_7_Strassen", "2x2x2_7_Winograd"):
        for small in ((1, 1, 2), (1, 2, 1), (2, 1, 1)):
            out[f"{stem}_kron_{''.join(map(str, small))}"] = kron(O.triple(stem), naive(*small))
    out["2x2x2_7_DPS-integral-12.0662_kron_112"] = kron(O.triple("2x2x2_7_DPS-integral-12.0662"), naive(1, 1, 2))
    out["2x2x2_7_DPS-intermediate-12.0695_kron_112"] = kron(O.triple("2x2x2_7_DPS-intermediate-12.0695"), naive(1, 1, 2))
    for mkn in ((1, 2, 2), (2, 3, 4), (2, 2, 8), (5, 5, 5)):
        out["naive_%dx%dx%d" % mkn] = naive(*mkn)
    return out


def is_algorithm(T):
    """The oracle's exact check over Q (mmcheck_q == 0) at every pair of unit vectors: the triple computes a bilinear map, so this
    proves it is a <m,k,n> matrix-multiplication algorithm.  With common denominators beyond 2^31 the oracle's int64 rationals
    overflow, so those triples are checked the same way modulo two primes instead."""
    m, k, n = O.LRP2MM(*T)
    eye_a, eye_b = np.eye(m * k, dtype=np.int64), np.eye(k * n, dtype=np.int64)
    pairs = [(i, j) for i in range(m * k) for j in range(k * n)]
    if max(O.lcm_den(M) for M in T) < 2 ** 31:
        return all(O.mmcheck_q(*T, eye_a[i], eye_b[j]) == 0 for i, j in pairs)
    return all(O.mmcheck_modp(p, *T, eye_a[i], eye_b[j]) == 0 for p in (2147483647, 2147483629) for i, j in pairs)


def scaled(T, dtype=np.int32):
    """(shape, (L, R, P) integer images, (denL, denR, denP)) for the C ABI."""
    (Li, dl), (Ri, dr), (Pi, dp) = (O.scaled_int(M) for M in T)
    return O.LRP2MM(*T), (Li.astype(dtype), Ri.astype(dtype), Pi.astype(dtype)), (dl, dr, dp)
