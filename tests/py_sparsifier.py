"""An INDEPENDENT restatement, in plain Python on `fractions.Fraction` / integers mod p, of the sparsifier pipeline
(include/plinopt_sparsify.inl: blockSparsifier :666-748, sparseAlternate :609-661, SparseFactor :473-513, localSparsifier :205-347,
testLinComb :166-197, FactorDiagonals :354-375, sparseLU/ILU :523-604, augment :20-35) with the documented stand-ins for the
LinBox routines that are not in the reference tree (DESIGN.md "pivot rule").

Test infrastructure only.  It shares no code with oracle/plo_oracle.cpp (C++) nor with the product's host layer: different
language, dense lists of Python objects, a brute-force quad loop (numpy on integer images, candidates visited in decreasing
key order).  tests/golden/sparsifier_goldens.json is generated from it (tests/golden/make_sparsifier_goldens.py); the oracle, the
product and this file must all agree on those (CoB, Res) pairs -- three independent routes to the same answer.
"""
import math
from fractions import Fraction

import numpy as np

COEFFICIENT_SEARCH = 11  # include/plinopt_sparsify.h:36-38


# ---- fields ---------------------------------------------------------------------------------------------------------
class QQ:
    p = 0

    def elt(self, num, den=1):
        return Fraction(num, den)

    def canon(self, a):
        return a

    def is_zero(self, a):
        return a == 0

    def add(self, a, b):
        return a + b

    def sub(self, a, b):
        return a - b

    def mul(self, a, b):
        return a * b

    def div(self, a, b):
        return a / b

    def inv(self, a):
        return 1 / a

    def neg(self, a):
        return -a

    def raw_neg(self, a):
        return -a

    def from_int(self, i):
        return Fraction(i)

    def less(self, a, b):
        return a < b


class Zp:
    """Elements are plain ints; field results are canonical in [0, p) while -r and the integers 2, 3, ... of the coefficient list stay
    un-reduced, as Givaro::Integer elements do in the reference (SURVEY.md section 9, Q3)."""

    def __init__(self, p):
        self.p = p

    def elt(self, num, den=1):
        return (num % self.p) * pow(den % self.p, -1, self.p) % self.p

    def canon(self, a):
        return a % self.p

    def is_zero(self, a):
        return a % self.p == 0

    def add(self, a, b):
        return (a + b) % self.p

    def sub(self, a, b):
        return (a - b) % self.p

    def mul(self, a, b):
        return (a * b) % self.p

    def div(self, a, b):
        return a * pow(b % self.p, -1, self.p) % self.p

    def inv(self, a):
        return pow(a % self.p, -1, self.p)

    def neg(self, a):
        return (-a) % self.p

    def raw_neg(self, a):
        return -a

    def from_int(self, i):
        return i

    def less(self, a, b):
        return a < b


# ---- libstdc++ std::sort, restated (Q7: the prelude sorts rows by size with an unstable sort; ties follow the algorithm) ----
def std_sort(items, comp):
    """bits/stl_algo.h: introsort (median-of-three quicksort down to 16 elements) + final insertion sort; in place."""
    a = items
    n = len(a)
    if n < 2:
        return a

    def move_median_to_first(result, x, y, z):
        if comp(a[x], a[y]):
            if comp(a[y], a[z]):
                a[result], a[y] = a[y], a[result]
            elif comp(a[x], a[z]):
                a[result], a[z] = a[z], a[result]
            else:
                a[result], a[x] = a[x], a[result]
        elif comp(a[x], a[z]):
            a[result], a[x] = a[x], a[result]
        elif comp(a[y], a[z]):
            a[result], a[z] = a[z], a[result]
        else:
            a[result], a[y] = a[y], a[result]

    def unguarded_partition(first, last, pivot):
        while True:
            while comp(a[first], a[pivot]):
                first += 1
            last -= 1
            while comp(a[pivot], a[last]):
                last -= 1
            if not first < last:
                return first
            a[first], a[last] = a[last], a[first]
            first += 1

    def introsort_loop(first, last, depth):
        while last - first > 16:
            if depth == 0:
                raise NotImplementedError("heapsort fallback of std::sort (never reached for the sizes of this path)")
            depth -= 1
            mid = first + (last - first) // 2
            move_median_to_first(first, first + 1, mid, last - 1)
            cut = unguarded_partition(first + 1, last, first)
            introsort_loop(cut, last, depth)
            last = cut

    def unguarded_linear_insert(last):
        val = a[last]
        nxt = last - 1
        while comp(val, a[nxt]):
            a[last] = a[nxt]
            last = nxt
            nxt -= 1
        a[last] = val

    def insertion_sort(first, last):
        for i in range(first + 1, last):
            if comp(a[i], a[first]):
                val = a[i]
                a[first + 1:i + 1] = a[first:i]
                a[first] = val
            else:
                unguarded_linear_insert(i)

    introsort_loop(0, n, 2 * (n.bit_length() - 1))
    if n > 16:
        insertion_sort(0, 16)
        for i in range(16, n):
            unguarded_linear_insert(i)
    else:
        insertion_sort(0, n)
    return a


# ---- dense helpers --------------------------------------------------------------------------------------------------
def transpose(M):
    return [list(r) for r in zip(*M)]


def identity(F, n):
    return [[F.from_int(1) if i == j else F.from_int(0) for j in range(n)] for i in range(n)]


def density(F, M):
    return sum(1 for row in M for v in row if not F.is_zero(v))


def matmul(F, A, B):
    out = [[F.from_int(0)] * len(B[0]) for _ in A]
    for i, row in enumerate(A):
        for t, a in enumerate(row):
            if F.is_zero(a):
                continue
            for j, b in enumerate(B[t]):
                if not F.is_zero(b):
                    out[i][j] = F.add(out[i][j], F.mul(a, b))
    return out


def rank(F, M):
    A = [list(r) for r in M]
    rk = 0
    cols = len(A[0]) if A else 0
    for c in range(cols):
        piv = next((i for i in range(rk, len(A)) if not F.is_zero(A[i][c])), None)
        if piv is None:
            continue
        A[rk], A[piv] = A[piv], A[rk]
        ip = F.inv(A[rk][c])
        for i in range(rk + 1, len(A)):
            if not F.is_zero(A[i][c]):
                mlt = F.mul(A[i][c], ip)
                A[i] = [F.sub(x, F.mul(mlt, y)) for x, y in zip(A[i], A[rk])]
        rk += 1
    return rk


def inverse(F, M):
    n = len(M)
    A = [list(r) + [F.from_int(1) if i == j else F.from_int(0) for j in range(n)] for i, r in enumerate(M)]
    for c in range(n):
        piv = next(i for i in range(c, n) if not F.is_zero(A[i][c]))
        A[c], A[piv] = A[piv], A[c]
        ip = F.inv(A[c][c])
        A[c] = [F.mul(x, ip) for x in A[c]]
        for i in range(n):
            if i != c and not F.is_zero(A[i][c]):
                mlt = A[i][c]
                A[i] = [F.sub(x, F.mul(mlt, y)) for x, y in zip(A[i], A[c])]
    return [row[n:] for row in A]


# ---- the documented pivot rule (stand-in for QLUPin) ------------------------------------------------------------------
def eliminate(F, A):
    """Step k: the remaining row with the fewest non-zeroes (first among ties, empty rows skipped) is swapped into place; its
    pivot is the entry whose column has the fewest non-zeroes among the remaining rows (first among ties).  A = Pr^T L U."""
    m, n = len(A), len(A[0])
    U = [list(r) for r in A]
    L = identity(F, m)
    rowperm = list(range(m))
    pivcol = []
    for k in range(m):
        sizes = [(sum(1 for v in U[i] if not F.is_zero(v)), i) for i in range(k, m)]
        cand = [(s, i) for s, i in sizes if s > 0]
        if not cand:
            break
        best = min(cand)[1]  # smallest size, then lowest position
        if best != k:
            U[k], U[best] = U[best], U[k]
            for j in range(k):
                L[k][j], L[best][j] = L[best][j], L[k][j]
            rowperm[k], rowperm[best] = rowperm[best], rowperm[k]
        pc = min((sum(1 for i in range(k, m) if not F.is_zero(U[i][j])), j) for j in range(n) if not F.is_zero(U[k][j]))[1]
        pivcol.append(pc)
        ip = F.inv(U[k][pc])
        for i in range(k + 1, m):
            if F.is_zero(U[i][pc]):
                continue
            mlt = F.mul(U[i][pc], ip)
            L[i][k] = mlt
            U[i] = [F.sub(x, F.mul(mlt, y)) if not F.is_zero(y) else x for x, y in zip(U[i], U[k])]
    return U, L, rowperm, pivcol


def nullspace_vector(F, N):
    """Stand-in for column 0 of nullspacebasisin (:235-239): first non-pivot column set to one, back substitution."""
    n = len(N[0])
    U, _, _, pivcol = eliminate(F, N)
    free = [j for j in range(n) if j not in pivcol]
    x = [F.from_int(0)] * n
    if not free:
        return x
    x[free[0]] = F.from_int(1)
    for kk in range(len(pivcol) - 1, -1, -1):
        s = F.from_int(0)
        for j in range(n):
            if j != pivcol[kk] and not F.is_zero(U[kk][j]) and not F.is_zero(x[j]):
                s = F.add(s, F.mul(U[kk][j], x[j]))
        x[pivcol[kk]] = F.neg(F.div(s, U[kk][pivcol[kk]]))
    return x


def sparse_lu(F, A, sparsity):
    U, L, rowperm, _ = eliminate(F, A)
    if density(F, U) >= sparsity:
        return None
    m = len(A)
    C = [[F.from_int(0)] * m for _ in range(m)]
    for k in range(m):
        C[rowperm[k]] = list(L[k])
    return C, U


def factor_diagonals(F, TCoB, TM):
    """:354-375; the most frequent value of a row, the smallest one (std::map order) among equally frequent (Q18)."""
    from collections import Counter
    for i, row in enumerate(TM):
        cnt = Counter(v for v in row if not F.is_zero(v))
        if not cnt:
            continue
        top = max(cnt.values())
        r = min(k for k, c in cnt.items() if c == top)
        if F.canon(r) != F.canon(F.from_int(1)):
            TM[i] = [F.div(v, r) if not F.is_zero(v) else v for v in row]
            TCoB[i] = [F.div(v, r) if not F.is_zero(v) else v for v in TCoB[i]]


def coefficients(F, TM, maxnumcoeff):
    """:20-35, :256-268 -- {0, 1, -1}, then r, -r, 1/r, -1/r for every stored entry r that is new, then 2, 3, ...; truncated."""
    C = [F.from_int(0), F.from_int(1), F.raw_neg(F.from_int(1))]

    def augment(r):
        if any(type(x) is type(r) and x == r for x in C):
            return
        t = F.inv(r)
        C.extend([r, F.raw_neg(r), t, F.neg(t)])
    for row in TM:
        for v in row:
            if not F.is_zero(v):
                augment(v)
    i = 2
    while len(C) < maxnumcoeff:
        augment(F.from_int(i))
        i += 1
    return C[:maxnumcoeff]


# ---- localSparsifier (:205-347) with a brute-force quad loop -----------------------------------------------------------
def integer_images(F, TM, Coeffs):
    """Zero patterns are invariant under scaling the columns of TM and the whole coefficient list: integer matrices for numpy
    (int64 when the products provably fit, Python integers otherwise)."""
    if F.p:  # products of two residues fit int64 for p <= 2^31; Python integers above
        dt = np.int64 if F.p <= 2 ** 31 else object
        return np.array([[F.canon(v) for v in row] for row in TM], dtype=dt), np.array([F.canon(c) for c in Coeffs], dtype=dt)
    cols = []
    for j in range(len(TM[0])):
        l = 1
        for i in range(len(TM)):
            l = l * TM[i][j].denominator // math.gcd(l, TM[i][j].denominator)
        cols.append([int(TM[i][j] * l) for i in range(len(TM))])
    l = 1
    for c in Coeffs:
        l = l * c.denominator // math.gcd(l, c.denominator)
    cf = [int(c * l) for c in Coeffs]
    small = 4 * max(abs(v) for col in cols for v in col) * max(abs(v) for v in cf) < 2 ** 62
    dt = np.int64 if small else object
    return np.array(cols, dtype=dt).T, np.array(cf, dtype=dt)


def local_sparsifier(F, TCoB, TM, maxnumcoeff, trace=None):
    n, m = len(TM), len(TM[0])
    LCoB = [[F.from_int(0)] * n for _ in range(n)]
    rnHw = cnHw = -1
    if n > 1:
        order = [(sum(1 for i in range(n) if not F.is_zero(TM[i][j])), j) for j in range(m)]
        std_sort(order, lambda a, b: a[0] > b[0])
        N = [[TM[i][j] for i in range(n)] for _, j in order]
        while N and rank(F, N) == n:
            N.pop()
        if N:
            x = nullspace_vector(F, N)
            LCoB[0] = [v if not F.is_zero(v) else F.from_int(0) for v in x]
            cnHw = sum(1 for v in LCoB[0] if not F.is_zero(v))  # non-zeroes (sic, :242)
            v = [sum((F.mul(LCoB[0][i], TM[i][j]) for i in range(n)), F.from_int(0)) for j in range(m)]
            rnHw = sum(1 for s in v if F.is_zero(s))
    Coeffs = coefficients(F, TM, maxnumcoeff)
    c = len(Coeffs)
    tm_int, cf_int = integer_images(F, TM, Coeffs)
    for block in range((n + 3) // 4):
        off = 4 * block
        nact = min(4, n - off)
        # score of every candidate, once: index = ((i*c + j)*c + k)*c + l, l fastest; positions beyond n are truncated (Q4)
        idx = np.arange(c ** 4)
        digits = [(idx // c ** (3 - t)) % c for t in range(4)]
        if F.p:
            v = sum(np.outer(cf_int[digits[t]], tm_int[off + t]) % F.p for t in range(nact)) % F.p
        else:
            v = sum(np.outer(cf_int[digits[t]], tm_int[off + t]) for t in range(nact))
        rl = (v == 0).sum(axis=1).astype(np.int64)
        cl = (n - nact) + sum((cf_int[digits[t]] == 0).astype(np.int64) for t in range(nact))
        order = np.lexsort((idx, -cl, -rl))  # decreasing (rl, cl), then increasing index: strict '>' acceptance = first maximiser
        for num in range(nact):
            row = off + num
            weight = (-1, -1)
            found = block == 0 and num == 0
            if found:
                weight = (rnHw, cnHw)
            for e in order:
                e = int(e)
                if (int(rl[e]), int(cl[e])) <= weight:
                    break
                w = [F.from_int(0)] * n
                for t in range(nact):
                    w[off + t] = Coeffs[int(digits[t][e])]
                cand = [list(r) for r in LCoB[:row]] + [w]
                if rank(F, cand) > row:
                    LCoB[row] = w
                    weight = (int(rl[e]), int(cl[e]))
                    found = True
                    if trace is not None:
                        trace.append((block, num, weight[0], weight[1], e, c))
                    break
            q = 0
            while not found:  # canonical fallback :317-326
                w = [F.from_int(0)] * n
                w[q] = F.from_int(1)
                if rank(F, [list(r) for r in LCoB[:row]] + [w]) > row:
                    LCoB[row] = w
                    found = True
                q += 1
    return matmul(F, LCoB, TCoB), matmul(F, LCoB, TM)


def sparse_factor(F, TICoB, TM, start, increment, threshold):
    s2 = density(F, TM)
    numcoeffs = start
    while True:
        ss = s2
        TICoB, TM = local_sparsifier(F, TICoB, TM, numcoeffs)
        factor_diagonals(F, TICoB, TM)
        s2 = density(F, TM)
        if numcoeffs < threshold:
            numcoeffs += increment
        if not s2 < ss:
            return TICoB, TM


def sparse_alternate(F, M, maxnumcoeff):
    TM = transpose(M)
    TICoB = identity(F, len(M[0]))
    factor_diagonals(F, TICoB, TM)
    lu = sparse_lu(F, TM, density(F, TM))
    if lu is not None:  # sparseILU :576-604
        QL, TM = lu
        TICoB = matmul(F, inverse(F, QL), TICoB)
    TICoB, TM = sparse_factor(F, TICoB, TM, 3, 4, COEFFICIENT_SEARCH)
    TICoB, TM = sparse_factor(F, TICoB, TM, maxnumcoeff, 1, maxnumcoeff)
    return transpose(inverse(F, TICoB)), transpose(TM)


def block_sparsifier(F, M, blocksize=4, maxnumcoeff=COEFFICIENT_SEARCH, initial_elimination=True):
    """-> (CoB, Res) with M == Res . CoB."""
    M = [[F.elt(v.numerator, v.denominator) if isinstance(v, Fraction) else F.elt(v) for v in row] for row in M]
    if blocksize <= 1:
        return sparse_alternate(F, M, maxnumcoeff)
    m, n = len(M), len(M[0])
    L = identity(F, n)
    A = M
    reduced = False
    if initial_elimination:
        U = transpose(M)
        lu = sparse_lu(F, U, density(F, U))
        if lu is not None:
            L, U = lu
            A = transpose(U)
            reduced = True
    Res = [[F.from_int(0)] * n for _ in range(m)]
    CoB = [[F.from_int(0)] * n for _ in range(n)]
    TCoB = [[F.from_int(0)] * n for _ in range(n)]
    for c0 in range(0, n, blocksize):
        w = min(blocksize, n - c0)
        C, R = sparse_alternate(F, [row[c0:c0 + w] for row in A], maxnumcoeff)
        for i in range(m):
            Res[i][c0:c0 + w] = R[i]
        if reduced:
            B = matmul(F, [row[c0:c0 + w] for row in L], transpose(C))
            for i in range(n):
                TCoB[i][c0:c0 + w] = B[i]
        else:
            for i in range(w):
                CoB[c0 + i][c0:c0 + w] = C[i]
    if reduced:
        CoB = transpose(TCoB)
    return [[F.canon(v) for v in row] for row in CoB], [[F.canon(v) for v in row] for row in Res]
