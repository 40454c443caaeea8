"""Host-side data plumbing for Hopcroft-Musinski (HM) matrices: the SMS text
format of the reference (data/README.md:10-17: optional '#' lines, header
`rows cols R|M`, 1-based `i j value` with value = integer or a/b, terminator
`0 0 0`), LCD scaling to the integer arrays the C ABI takes, CSR mod p."""
import json
import lzma
import math
import os
import re
from fractions import Fraction

import numpy as np


def _read_sms(path_or_lines, parse, zero):
    """The loop of every SMS reader: -> list of rows of parse(token), `zero` where no entry is given."""
    if isinstance(path_or_lines, str):
        with open(path_or_lines) as f:
            lines = f.readlines()
    else:
        lines = list(path_or_lines)
    rows = cols = None
    M = None
    for line in lines:
        s = line.strip()
        if not s or s.startswith("#"):
            continue
        t = s.split()
        if rows is None:
            rows, cols = int(t[0]), int(t[1])
            M = [[zero] * cols for _ in range(rows)]
            continue
        i, j = int(t[0]), int(t[1])
        if i == 0 and j == 0:
            break
        M[i - 1][j - 1] = parse(t[2])
    if M is None:
        raise ValueError("empty SMS stream")
    return M


def read_sms(path_or_lines):
    """-> list of rows of Fraction."""
    return _read_sms(path_or_lines, Fraction, Fraction(0))


def write_sms(M, path=None, fmt=str):
    """LinBox FileFormat(5) shape: `rows cols M`, entries row-major, `0 0 0` (src/orbiter.cpp:346-348).  `fmt` writes a non-zero
    entry."""
    out = [f"{len(M)} {len(M[0])} M"]
    for i, row in enumerate(M):
        for j, v in enumerate(row):
            if v != 0:
                out.append(f"{i + 1} {j + 1} {fmt(v)}")
    out.append("0 0 0")
    text = "\n".join(out) + "\n"
    if path:
        with open(path, "w") as f:
            f.write(text)
    return text


# An entry a + b.X of Q(sqrt d), X^2 = d (`-P "X^2-d"`): `q`, `qX`, `X`, `-X`, `q+qX`, `q-qX`, the coefficient of X omitted for +-1.
# The reference's `*-X_*` files and its reader are not available here: the grammar is a restatement (DESIGN.md 5.1).
_Q = r"[+-]?\d+(?:/\d+)?"
_QUAD = re.compile(rf"(?P<a>{_Q})|(?P<x>{_Q}|[+-]?)X|(?P<a2>{_Q})(?P<s>[+-])(?P<b2>\d+(?:/\d+)?)?X")


def parse_quad(tok):
    """'1/2-X' -> (Fraction(1, 2), Fraction(-1))."""
    m = _QUAD.fullmatch(tok)
    if m is None:
        raise ValueError(f"cannot parse matrix entry {tok!r} as a + bX")
    if m["a"] is not None:
        return Fraction(m["a"]), Fraction(0)
    if m["x"] is not None:
        return Fraction(0), Fraction(-1 if m["x"] == "-" else 1 if m["x"] in ("", "+") else m["x"])
    b = Fraction(m["b2"] or 1)
    return Fraction(m["a2"]), -b if m["s"] == "-" else b


def format_quad(a, b):
    """The forms parse_quad reads: `a`, `bX` (`X`, `-X`), `a+bX`, `a-|b|X`."""
    if b == 0:
        return str(a)
    coef = "" if abs(b) == 1 else str(abs(b))
    if a == 0:
        return ("-" if b < 0 else "") + coef + "X"
    return f"{a}{'-' if b < 0 else '+'}{coef}X"


def read_sms_quad(path_or_lines):
    """-> (A, B): the rational parts and the parts in X, lists of rows of Fraction."""
    M = _read_sms(path_or_lines, parse_quad, (Fraction(0), Fraction(0)))
    return [[e[0] for e in row] for row in M], [[e[1] for e in row] for row in M]


def write_sms_quad(M, path=None):
    """SMS of a pair (A, B) of lists of rows of Fraction, entries A + B.X."""
    A, B = M
    return write_sms([list(zip(ra, rb)) for ra, rb in zip(A, B)], path, fmt=lambda e: format_quad(*e))


def load_fixture(stem, json_path=None):
    """(L, R, P) Fraction matrices of a triple stored in tests/golden/hm_matrices.json (data fixture)."""
    if json_path is None:
        json_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "hm_matrices.json")
    with open(json_path) as f:
        d = json.load(f)
    out = []
    for x in "LRP":
        e = d[f"{stem}_{x}"]
        M = [[Fraction(0)] * e["cols"] for _ in range(e["rows"])]
        for i, j, v in e["entries"]:
            M[i][j] = Fraction(v)
        out.append(M)
    return tuple(out)


def lcd(M):
    l = 1
    for row in M:
        for v in row:
            l = l * v.denominator // math.gcd(l, v.denominator)
    return l


def scaled(M, dtype=np.int64):
    """(integer array of M * lcd, lcd)."""
    d = lcd(M)
    return np.array([[int(v * d) for v in row] for row in M], dtype=dtype), d


def LRP2MM(L, R, P):
    """include/plinopt_library.h:177-181."""
    n = int(math.sqrt(len(R[0]) * len(P) // len(L[0])))
    return len(P) // n, len(R[0]) // n, n


def csr_modp(M, p):
    """(rows, cols, ptr, col, val) with val = a * b^-1 mod p (src/MMchecker.cpp rebind to Modular)."""
    ptr = [0]; col = []; val = []
    for row in M:
        for j, v in enumerate(row):
            if v != 0:
                x = (v.numerator % p) * pow(v.denominator % p, -1, p) % p
                if x:
                    col.append(j); val.append(x)
        ptr.append(len(col))
    return (len(M), len(M[0]), np.array(ptr, dtype=np.int64), np.array(col, dtype=np.int32), np.array(val, dtype=np.uint32))


def strip_modulus(q):
    """src/MMchecker.cpp:123-126, src/orbiter.cpp:419-422: drop the factors of 2, 1 -> 2."""
    while q % 2 == 0 and q > 0:
        q >>= 1
    return 2 if q == 1 else q


LARGE_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "large", "32x32x32_15096.npz")


def save_large(path, arrays):
    """Stores CSR matrices given as {X_shape, X_ptr, X_col, X_num, X_den} (rational entries num/den, columns ascending in each
    row) in a compact form that load_large() turns back into the same arrays.  Each matrix lists its non-zeroes along its longer
    dimension (row-major when rows >= cols, else column-major), three bytes per entry: the gap to the previous entry's linear
    index (uint16, little-endian) and the entry's position in the table X_values of the matrix's distinct (num, den) pairs; the
    byte stream is xz-compressed into X_entries.  For 32x32x32_15096 this takes 0.2 MB against 2 MB for the plain CSR."""
    out = {}
    for x in sorted({k.split("_")[0] for k in arrays}):
        rows, cols = (int(v) for v in arrays[f"{x}_shape"])
        ptr, col = np.asarray(arrays[f"{x}_ptr"], np.int64), np.asarray(arrays[f"{x}_col"], np.int64)
        row = np.repeat(np.arange(rows, dtype=np.int64), np.diff(ptr))
        lin = row * cols + col if rows >= cols else col * rows + row
        order = np.argsort(lin, kind="stable")
        gap = np.diff(lin[order], prepend=-1)
        pairs = np.stack([np.asarray(arrays[f"{x}_num"], np.int64), np.asarray(arrays[f"{x}_den"], np.int64)], axis=1)[order]
        values, code = np.unique(pairs, axis=0, return_inverse=True)
        if len(gap) and (gap.min() < 1 or gap.max() > 0xFFFF) or len(values) > 256:
            raise ValueError(f"{x} does not fit the compact encoding")
        rec = np.stack([gap & 0xFF, gap >> 8, code.reshape(-1)], axis=1).astype(np.uint8)
        out.update({f"{x}_shape": np.array([rows, cols], dtype=np.int64), f"{x}_values": values,
                    f"{x}_entries": np.frombuffer(lzma.compress(rec.tobytes(), preset=9 | lzma.PRESET_EXTREME), dtype=np.uint8)})
    np.savez(path, **out)


def load_large(path=None):
    """The regenerated 32x32x32_15096 triple (tools/regen_32x32x32.py) as row-major CSR arrays with rational values:
    {X_shape, X_ptr (int64), X_col, X_num, X_den (int32)} for X in L, R, P, or None when the file is absent."""
    path = LARGE_PATH if path is None else path
    if not os.path.exists(path):
        return None
    z = np.load(path)
    out = {}
    for x in sorted({k.split("_")[0] for k in z.files}):
        rows, cols = (int(v) for v in z[f"{x}_shape"])
        rec = np.frombuffer(lzma.decompress(z[f"{x}_entries"].tobytes()), dtype=np.uint8).reshape(-1, 3).astype(np.int64)
        lin = np.cumsum(rec[:, 0] | (rec[:, 1] << 8)) - 1
        num, den = z[f"{x}_values"][rec[:, 2]].T
        if rows >= cols:
            row, col = np.divmod(lin, cols)
        else:
            col, row = np.divmod(lin, rows)
            order = np.lexsort((col, row))
            row, col, num, den = row[order], col[order], num[order], den[order]
        ptr = np.zeros(rows + 1, dtype=np.int64)
        np.cumsum(np.bincount(row, minlength=rows), out=ptr[1:])
        out.update({f"{x}_shape": z[f"{x}_shape"], f"{x}_ptr": ptr, f"{x}_col": col.astype(np.int32),
                    f"{x}_num": num.astype(np.int32), f"{x}_den": den.astype(np.int32)})
    return out


def load_large_csr(p, path=None):
    """The regenerated 32x32x32_15096 triple (tools/regen_32x32x32.py) reduced mod p:
    returns (mkn, r, (L, R, P) CSR tuples) or None when the file is absent."""
    z = load_large(path)
    if z is None:
        return None
    out = []
    for x in "LRP":
        rows, cols = (int(v) for v in z[f"{x}_shape"])
        num = z[f"{x}_num"].astype(np.int64) % p
        den = z[f"{x}_den"].astype(np.int64) % p
        inv = {int(d): pow(int(d), -1, p) for d in np.unique(den)}
        val = (num * np.array([inv[int(d)] for d in den], dtype=np.int64)) % p if p < (1 << 31) else np.array([(int(a) * inv[int(d)]) % p for a, d in zip(num, den)], dtype=np.int64)
        out.append((rows, cols, z[f"{x}_ptr"].astype(np.int64), z[f"{x}_col"].astype(np.int32), val.astype(np.uint32)))
    return (32, 32, 32), 15096, tuple(out)
