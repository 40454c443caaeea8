"""CPU tests of the `-P "X^2-d"` file layer: SMS entries a + bX (hm.read_sms_quad / hm.write_sms_quad and the C++ reader of the
CLIs), the refusals of the CLIs, and the argument checks of plo_mmchecker_quad, plo_orbiter_quad and plo_orbiter_progress_quad
before any device work."""
import os
import subprocess
from fractions import Fraction

import pytest

import oracle_lib as O
from plinopt_b200 import capi, hm
from test_quadratic_host import FX, zeros_like

BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin")
CLIS = ("MMchecker", "orbiter", "growthfactor")


def write_quad(tmp_path, stem, T):
    paths = []
    for x, M in zip("LRP", T):
        p = tmp_path / f"{stem}_{x}.sms"
        hm.write_sms_quad(M, str(p))
        paths.append(str(p))
    return paths


def run(exe, args):
    return subprocess.run([os.path.join(BIN, exe)] + args, capture_output=True, text=True, timeout=120)


def form(tok):
    a, b = hm.parse_quad(tok)
    if b == 0:
        return "q"
    if a == 0:
        return "X" if abs(b) == 1 else "qX"
    return "q+qX" if b > 0 else "q-qX"


# one entry of each form, with and without unit coefficients of X (the FX fixtures never mix both parts in one entry)
MIXED = ([[Fraction(1, 2), Fraction(0), Fraction(-3), Fraction(2), Fraction(0), Fraction(0), Fraction(-1, 2)]],
         [[Fraction(0), Fraction(1, 2), Fraction(0), Fraction(3, 4), Fraction(-1), Fraction(1), Fraction(-1)]])


@pytest.mark.parametrize("name", sorted(FX) + ["mixed"])
def test_round_trip(name):
    pairs = [MIXED] if name == "mixed" else FX[name][1]
    for A, B in pairs:
        text = hm.write_sms_quad((A, B))
        assert hm.read_sms_quad(text.splitlines()) == ([list(r) for r in A], [list(r) for r in B])


def test_writer_emits_every_form():
    text = hm.write_sms_quad(MIXED)
    entries = [line.split()[2] for line in text.splitlines()[1:-1]]
    assert entries == ["1/2", "1/2X", "-3", "2+3/4X", "-X", "X", "-1/2-X"]
    assert {form(e) for e in entries} == {"q", "qX", "X", "q+qX", "q-qX"}


@pytest.mark.parametrize("tok,want", [("3", (3, 0)), ("-1/2", (Fraction(-1, 2), 0)), ("1/2X", (0, Fraction(1, 2))), ("-3X", (0, -3)), ("X", (0, 1)),
                                      ("-X", (0, -1)), ("1/2-X", (Fraction(1, 2), -1)), ("2+3/4X", (2, Fraction(3, 4))), ("-1+X", (-1, 1))])
def test_entry_forms(tok, want):
    assert hm.parse_quad(tok) == tuple(Fraction(v) for v in want)
    assert hm.format_quad(*hm.parse_quad(tok)) == tok


@pytest.mark.parametrize("tok", ["X2", "1/2XX", "1+2+X", "+-X", "1.5X", "Y"])
def test_malformed_entries_are_refused(tok):
    with pytest.raises(ValueError):
        hm.parse_quad(tok)
    text = f"1 1 M\n1 1 {tok}\n0 0 0\n"
    with pytest.raises(ValueError):
        hm.read_sms_quad(text.splitlines())


def test_rational_file_reads_identically():
    for M in O.triple("2x2x2_7_DPS-smallrat-12.2034"):
        text = hm.write_sms(M).splitlines()
        assert hm.read_sms_quad(text) == (hm.read_sms(text), zeros_like(M))


@pytest.mark.parametrize("tok", ["X2", "1/2XX", "1+2+X"])
def test_clis_refuse_malformed_entries(tmp_path, tok):
    files = write_quad(tmp_path, "dps", FX["DPS-accurate"][1])
    bad = tmp_path / "bad_L.sms"
    bad.write_text(f"1 1 M\n1 1 {tok}\n0 0 0\n")
    for exe in CLIS:
        p = run(exe, ["-P", "X^2-3", str(bad)] + files[1:])
        assert p.returncode == 255 and f"cannot parse matrix entry '{tok}'" in p.stderr, (exe, p.stderr)


def test_clis_refuse_what_is_out_of_scope(tmp_path):
    files = write_quad(tmp_path, "dps", FX["DPS-accurate"][1])
    for exe in CLIS:
        p = run(exe, ["-P", "X^3-2"] + files)
        assert p.returncode == 255 and "only X^2-d" in p.stderr, (exe, p.stderr)
        p = run(exe, ["-P", "X^2-3", "-m", "7"] + files)
        assert p.returncode == 255 and "-P cannot be combined with -m/-q/-r" in p.stderr, (exe, p.stderr)
        p = run(exe, ["-I", "X^2-3"] + files)
        assert p.returncode == 255 and "-I is out of scope" in p.stderr, (exe, p.stderr)
        p = run(exe, files)  # entries in X without -P
        assert p.returncode == 255 and "entries in X need -P" in p.stderr, (exe, p.stderr)
        p = run(exe, ["-P", "X^2 - 4"] + files)
        assert p.returncode == (capi.E_ARG & 0xFF) and "perfect square" in p.stderr, (exe, p.stderr)


@pytest.mark.skipif(capi.device_count() > 0, reason="checks the no-device behaviour")
def test_clis_fail_loudly_without_a_device(tmp_path):
    files = write_quad(tmp_path, "dps", FX["DPS-accurate"][1])
    for exe in CLIS:
        for poly in ("X^2-3", "X^2 + 1"):
            if exe == "growthfactor" and "+" in poly:
                continue  # G2 needs d > 0
            p = run(exe, ["-P", poly] + files)
            assert p.returncode == (capi.E_NODEVICE & 0xFF) and "no CUDA device" in p.stderr, (exe, poly, p.stderr)


def quad_calls(d, T):
    return (lambda: capi.mmchecker_quad(d, *T),
            lambda: capi.orbiter_quad(d, *T, measure=capi.MEASURE_NNZ),
            lambda: capi.orbiter_progress_quad(d, *T, measure=capi.MEASURE_NNZ))


def test_new_symbols_are_exported():
    L = capi.lib()
    for s in ("plo_mmchecker_quad", "plo_orbiter_quad", "plo_orbiter_progress_quad"):
        assert s in capi.SYMBOLS and hasattr(L, s)


@pytest.mark.parametrize("d", [0, 1, 4, 9, 1 << 40])
def test_perfect_squares_are_refused(d):
    for call in quad_calls(d, FX["DPS-accurate"][1]):
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == capi.E_ARG


def test_orbiter_growth_factor_needs_a_real_embedding():
    T = FX["2x2x2_7_Winograd_sqrt-3"][1]
    for call in (lambda: capi.orbiter_quad(-3, *T, measure=capi.MEASURE_G2), lambda: capi.orbiter_progress_quad(-3, *T, measure=capi.MEASURE_G2)):
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == capi.E_ARG


@pytest.mark.skipif(capi.device_count() > 0, reason="checks the no-device behaviour")
@pytest.mark.parametrize("name", ["DPS-accurate", "2x2x2_7_Winograd_sqrt-1"])
def test_quadratic_drivers_fail_loudly_without_a_device(name):
    d, T = FX[name]
    for call in quad_calls(d, T):
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == capi.E_NODEVICE
