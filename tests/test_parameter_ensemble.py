"""ensemble.parameter_sets: the ABCD parameter tables of a parameter ensemble as float64 [P, n_rows, 5] (host only),
4-column tables with m = 0, and its refusals."""

import numpy as np
import pytest


def test_one_array_and_a_sequence_of_tables():
    from xanthos_b200 import ensemble as ens
    rng = np.random.default_rng(0)
    a = rng.uniform(0.1, 0.9, (3, 7, 5))
    got = ens.parameter_sets(a, 7)
    assert got.dtype == np.float64 and got.shape == (3, 7, 5) and np.array_equal(got, a)
    assert got is not a                                          # the caller's array is not kept
    assert np.array_equal(ens.parameter_sets(list(a), 7), a)
    assert np.array_equal(ens.parameter_sets(tuple(t.tolist() for t in a), 7), a)
    assert np.array_equal(ens.parameter_sets(a.astype(np.float32), 7), a.astype(np.float32).astype(np.float64))


def test_four_column_tables_get_no_snow_melt():
    from xanthos_b200 import ensemble as ens
    rng = np.random.default_rng(1)
    four = rng.uniform(0.1, 0.9, (2, 4, 4))
    got = ens.parameter_sets(four, 4)
    assert got.shape == (2, 4, 5)
    assert np.array_equal(got[:, :, :4], four) and np.array_equal(got[:, :, 4], np.zeros((2, 4)))
    five = rng.uniform(0.1, 0.9, (4, 5))
    mixed = ens.parameter_sets([four[0], five], 4)
    assert np.array_equal(mixed[0], got[0]) and np.array_equal(mixed[1], five)


@pytest.mark.parametrize("sets,match", [
    (np.ones((2, 6, 5)), '6 rows'),
    ([np.ones((5, 5)), np.ones((4, 5))], 'parameter set 1 has 4 rows'),
    (np.ones((2, 5, 3)), '3 columns'),
    ([np.ones((5, 6))], '6 columns'),
    (np.ones((5, 5)), 'shape'),
    (np.ones((1, 2, 5, 5)), 'shape'),
    ([np.ones(5)] * 5, 'parameter set 0 has shape'),
    ([np.ones((1, 5, 5))], 'parameter set 0 has shape'),
    ([], 'no parameter set'),
    (np.ones((0, 5, 5)), 'no parameter set'),
])
def test_refusals(sets, match):
    from xanthos_b200 import ensemble as ens, _cuda as C
    with pytest.raises(C.ValidationException, match=match):
        ens.parameter_sets(sets, 5)
