"""GPU tests of the drop-in CLIs (same flags / streams / files as src/sparsifier.cpp, src/orbiter.cpp, src/MMchecker.cpp)."""
import os
import subprocess

import pytest

import oracle_lib as O
from plinopt_b200 import hm

pytestmark = pytest.mark.gpu
BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin")


def write_triple(tmp_path, stem):
    paths = []
    for x, M in zip("LRP", O.triple(stem)):
        p = tmp_path / f"{stem}_{x}.sms"
        hm.write_sms(M, str(p))
        paths.append(str(p))
    return paths


def test_sparsifier_cli_fdt_style(capi, tmp_path):
    """bin/FDT.sh:64-66: `sparsifier -c 5 f` and `sparsifier -q 7 -c 5 f` must print SUCCESS; -S output parses back to the oracle's CoB."""
    M = O.dense_fractions("2x2x2_7_DPS-smallrat-12.2034_L")
    f = tmp_path / "m.sms"
    hm.write_sms(M, str(f))
    for extra in ([], ["-q", "7"]):
        p = subprocess.run([os.path.join(BIN, "sparsifier"), "-S", "-c", "5"] + extra + [str(f)], capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr
        assert "SUCCESS: consistent factorization!" in p.stderr and "# [SPRF] linear combination coefficients:" in p.stderr
        CoB = hm.read_sms(p.stdout.splitlines())
        eC, eR, ok, _ = O.sparsifier(M, 7 if extra else 0, 4, 5, True)
        assert CoB == [[O.Fraction(v) for v in row] for row in eC]
    # stdin input and -c 4 (BASELINE config 1)
    p = subprocess.run([os.path.join(BIN, "sparsifier"), "-c", "4"], input=open(f).read(), capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "SUCCESS" in p.stderr and "7x4 by 4x4" in p.stderr


def test_orbiter_cli_writes_nnz_sms(capi, tmp_path):
    files = write_triple(tmp_path, "2x2x2_7_Winograd")
    p = subprocess.run([os.path.join(BIN, "orbiter"), "-g", "-O", "20000", "--seed", "77"] + files, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "# Init. ops:" in p.stderr and "# Search(20000):" in p.stderr and "Rdcd. opt" in p.stderr
    outs = [f.replace(".sms", ".nnz.sms") for f in files]
    Lj, Rg, hP = (hm.read_sms(o) for o in outs)
    assert O.growth_G2(Lj, Rg, hP) < 15.0  # Winograd (17.85) -> 14.83 point of its orbit
    q = subprocess.run([os.path.join(BIN, "MMchecker")] + outs, capture_output=True, text=True, timeout=300)
    assert q.returncode == 0 and "SUCCESS: correct 2x2x2" in q.stderr


def test_mmchecker_cli_exit_codes(capi, tmp_path):
    """Makefile:60-64 mmcheck targets + the error codes of src/MMchecker.cpp:65-71 / plinopt_library.inl:494,555."""
    s = write_triple(tmp_path, "2x2x2_7_Strassen")
    a = write_triple(tmp_path, "2x2x2_7_DPS-accurate")
    run = lambda args: subprocess.run([os.path.join(BIN, "MMchecker")] + args, capture_output=True, text=True, timeout=300)
    assert run(s).returncode == 0
    assert run(["-m", "513083"] + a).returncode == 0
    assert run(["-r", "1013", "2", "3"] + a).returncode == 0
    r = run(a)
    assert r.returncode == 1 and "ERROR, not a 2x2x2 MM algorithm" in r.stderr
    w = write_triple(tmp_path, "3x3x3_23_58")
    assert run([s[0], w[1], s[2]]).returncode == 2
    # -b is the reference's bit size of the random coordinates (src/MMchecker.cpp:95-97), --samples the number of points; over Q the
    # verdict is exact at those points and the CLI says modulo how many primes it was taken
    r = run(["-b", "8", "--samples", "5"] + w)
    assert r.returncode == 0 and "# over Q: 5 points of 8-bit coordinates, decided modulo" in r.stderr
    r = run(["-b", "64"] + w)
    assert r.returncode == 0 and "NOTE: -b 64" in r.stderr and "32 points of 32-bit coordinates" in r.stderr


def test_factorizer_cli(capi, tmp_path):
    """src/factorizer.cpp:139-206 flags; CoB on stdout (-S parses back), Alt + SUCCESS line on stderr, -k outside range -> -1."""
    M = O.dense_fractions("4x4x4_48_rational_L")
    f = tmp_path / "m.sms"
    hm.write_sms(M, str(f))
    exe = os.path.join(BIN, "factorizer")
    p = subprocess.run([exe, "-S", "-O", "300", "-s", "99", str(f)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "# [FCTZ] Initial profile:" in p.stderr and "SUCCESS: consistent factorization!" in p.stderr and "48x16 by 16x16" in p.stderr
    CoB = hm.read_sms(p.stdout.splitlines())
    ref = O.factor_sweep(M, 16, 99, 0, 300, matrices=True)
    assert CoB == ref["cob"]
    p = subprocess.run([exe, "-k", "20", "-O", "100", "-q", "513083", str(f)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "48x20 by 20x16" in p.stderr and "SUCCESS" in p.stderr
    p = subprocess.run([exe, "-V", "1", "-c", "5", "-O", "100", str(f)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "SUCCESS: consistent factorization!" in p.stderr
    p = subprocess.run([exe, "-k", "5", str(f)], capture_output=True, text=True, timeout=300)
    assert p.returncode == 255 and "inner dimension has to be between 16 and 48" in p.stderr


def test_orbiter_cli_modular(capi, tmp_path):
    """-m p: the reference runs Orbiter<0> over Z/pZ (src/orbiter.cpp:419-426); outputs are residues and pass MMchecker -m p."""
    files = write_triple(tmp_path, "2x2x2_7_DPS-accurate")
    p = subprocess.run([os.path.join(BIN, "orbiter"), "-m", "513083", "-O", "20000", "--seed", "3"] + files, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "SUCCESS: correct 2x2x2" in p.stderr and "# Search(20000):" in p.stderr
    if "Rdcd. opt" in p.stderr:
        outs = [f.replace(".sms", ".nnz.sms") for f in files]
        q = subprocess.run([os.path.join(BIN, "MMchecker"), "-m", "513083"] + outs, capture_output=True, text=True, timeout=300)
        assert q.returncode == 0 and "SUCCESS: correct 2x2x2" in q.stderr


def test_negater_and_rotater_cli(capi, tmp_path):
    """src/negater.cpp (L.neg.sms ...) and bin/rotater.sh (<stem>_left_L.sms ..., then MMchecker of the rotated algorithm)."""
    files = write_triple(tmp_path, "3x4x7_63_rational")
    p = subprocess.run([os.path.join(BIN, "negater")] + files, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "# NEGs:" in p.stderr and "# GCDs:" in p.stderr, p.stderr
    outs = [f.replace(".sms", ".neg.sms") for f in files]
    (eL, eR, eP), _ = O.negater(*O.triple("3x4x7_63_rational"))
    assert [hm.read_sms(o) for o in outs] == [eL, eR, eP]
    q = subprocess.run([os.path.join(BIN, "MMchecker")] + outs, capture_output=True, text=True, timeout=300)
    assert q.returncode == 0 and "SUCCESS: correct 3x4x7" in q.stderr
    p = subprocess.run([os.path.join(BIN, "rotater"), "-r"] + files, capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert p.returncode == 0 and "SUCCESS: correct 7x3x4" in p.stderr, p.stderr
    rot = [hm.read_sms(str(tmp_path / f"3x4x7_63_rational_right_{x}.sms")) for x in "LRP"]
    assert rot == O.rotater(*O.triple("3x4x7_63_rational"), right=True)


def test_mmchecker_cli_on_the_regenerated_32x32x32(capi, tmp_path):
    """`make largecheck` (Makefile:89-93) / BASELINE config 5 through the drop-in CLI: the 32x32x32_15096 triple (regenerated from the reference's .slp, written back
    as SMS with its rational coefficients) is a correct algorithm over Q-reduced-mod-p; a corrupted P is not."""
    import numpy as np
    z = hm.load_large()
    files = []
    for x in "LRP":
        rows, cols = (int(v) for v in z[f"{x}_shape"])
        ptr, col, num, den = z[f"{x}_ptr"], z[f"{x}_col"], z[f"{x}_num"], z[f"{x}_den"]
        ri = np.repeat(np.arange(rows), np.diff(ptr))
        f = tmp_path / f"32x32x32_15096_{x}.sms"
        with open(f, "w") as fh:
            fh.write(f"{rows} {cols} R\n")
            fh.write("\n".join(f"{i + 1} {c + 1} {n}" + (f"/{d}" if d != 1 else "") for i, c, n, d in zip(ri.tolist(), col.tolist(), num.tolist(), den.tolist())))
            fh.write("\n0 0 0\n")
        files.append(str(f))
    run = lambda args: subprocess.run([os.path.join(BIN, "MMchecker")] + args, capture_output=True, text=True, timeout=600)
    p = run(["-m", "2147483647"] + files)
    assert p.returncode == 0 and "SUCCESS: correct 32x32x32" in p.stderr, p.stderr[-500:]
    bad = tmp_path / "bad_P.sms"
    lines = open(files[2]).read().splitlines()
    i, c, v = lines[5].split()
    lines[5] = f"{i} {c} 5"
    bad.write_text("\n".join(lines) + "\n")
    q = run(["-m", "2147483647", files[0], files[1], str(bad)])
    assert q.returncode == 1 and "not a 32x32x32 MM algorithm" in q.stderr


def test_growthfactor_cli(capi, tmp_path):
    files = write_triple(tmp_path, "2x2x2_7_Strassen")
    p = subprocess.run([os.path.join(BIN, "growthfactor")] + files, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "# Norms of 2x2x2 Matrix-Multiplication:" in p.stderr and "## Ginfinf:\t12.000000" in p.stderr and "## G2:\t\t14.828427" in p.stderr
    bad = write_triple(tmp_path, "3x3x3_23_58")
    assert subprocess.run([os.path.join(BIN, "growthfactor"), files[0], bad[1], files[2]], capture_output=True, text=True, timeout=300).returncode == 2


def test_orbiter_cli_progress_lines_and_bitsize(capi, tmp_path):
    """'# Found opt:' records (src/orbiter.cpp:312-315), deterministic: the successive prefix minima in index order; the last one is the
    winner of the 'Rdcd. opt' line, every record improves on the one before, and they equal plo_orbiter_progress.  -b is the bit size of
    the coordinates of the MMchecker's random points (at most 32) and the NOTE says so."""
    import re
    files = write_triple(tmp_path, "3x3x3_23_58")
    p = subprocess.run([os.path.join(BIN, "orbiter"), "-b", "8", "-O", "300000", "--seed", "5"] + files, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert "NOTE: -b 8: 32 random points with 8-bit coordinates" in p.stderr
    recs = [(float(a), int(b), int(c), int(i)) for a, b, c, i in re.findall(r"# Found opt: ([0-9.]+)[<=][0-9.]+\t\{(\d+),(\d+)\}&\{\d+,\d+\}\t\[(\d+)/gpu\]", p.stderr)]
    assert len(recs) >= 2
    assert all(x[3] < y[3] and (x[1], x[2]) > (y[1], y[2]) for x, y in zip(recs, recs[1:]))
    win = re.search(r"Rdcd\. opt: ([0-9.]+)<[0-9.]+\t\{(\d+),(\d+)\}.*\[(\d+)\]", p.stderr)
    assert (int(win.group(2)), int(win.group(3)), int(win.group(4))) == recs[-1][1:]
    L, R, P = O.triple("3x3x3_23_58")
    api = capi.orbiter_progress(L, R, P, capi.MEASURE_NNZ, capi.MODE_PHILOX, 5, 300000)
    assert [(r["nnz"], r["nno"], r["index"]) for r in api] == [x[1:] for x in recs]
    # every record really is the minimum of its prefix: check the first two against the oracle's table of the prefix
    tab = O.orbit_sweep(L, R, P, 0, 1, 5, 0, api[1]["index"] + 1)
    keys = list(zip(tab["nnz"].tolist(), tab["nno"].tolist()))
    assert min(range(len(keys)), key=lambda i: (keys[i], i)) == api[1]["index"] and min(range(api[1]["index"]), key=lambda i: (keys[i], i)) == api[0]["index"]


def test_orbiter_cli_rejects_inner_dimension_mismatch(capi, tmp_path):
    """The reference only warns (src/orbiter.cpp:236-242) and then fails inside LinBox; the engine takes flat buffers, so it rejects
    the triple with fMMchecker's code 2 instead of reading past them."""
    s = write_triple(tmp_path, "2x2x2_7_Strassen")
    w = write_triple(tmp_path, "3x3x3_23_58")
    p = subprocess.run([os.path.join(BIN, "orbiter"), "-O", "10", s[0], w[1], s[2]], capture_output=True, text=True, timeout=300)
    assert p.returncode == 2 and "inner dimension mismatch" in p.stderr
