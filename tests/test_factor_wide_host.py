"""Factorizer on a wide matrix (fewer rows than columns): the inner-dimension check comes first, as in the reference
(plinopt_sparsify.inl:936-942), so `factorizer` returns -1 with the reference's message whatever the width.  That path
returns before any device call and runs without a GPU."""
import oracle_lib as O
from plinopt_b200 import capi


def test_wide_matrix_gets_the_inner_dimension_failure():
    M = O.dense_fractions("4x4x4_48_rational_P")  # 16 x 48 as stored
    assert (len(M), len(M[0])) == (16, 48)
    rc = capi.factorizer(M)[0]
    assert rc == -1
    assert capi.lib().plo_last_error().decode() == "Fail: inner dimension has to be between 48 and 16."
