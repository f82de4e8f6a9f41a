"""The ensemble runner's PET models on the host: the member keys of every model, lossless float32 transport of their
fields (shared arrays stay shared) and the configurations EnsembleStatics refuses before it touches a device."""

import numpy as np
import pytest


def test_forcing_fields_of_every_pet_model():
    from xanthos_b200 import ensemble as ens
    assert ens.forcing_fields('pm') == ens.FORCING
    assert ens.forcing_fields('hs') == ('hs_tas', 'hs_tmax', 'hs_tmin', 'precip', 'tmin')
    assert ens.forcing_fields('thornthwaite') == ('tair', 'precip', 'tmin')
    assert ens.forcing_fields('none') == ('pet', 'precip', 'tmin')
    assert ens.PET_MODELS == ('pm', 'hs', 'thornthwaite', 'none')


@pytest.mark.parametrize("name", ['hargreaves', 'PM', '', None])
def test_unknown_pet_model_refused(name):
    from xanthos_b200 import ensemble as ens, _cuda as C
    with pytest.raises(C.ValidationException, match='unknown PET model'):
        ens.forcing_fields(name)
    with pytest.raises(C.ValidationException, match='unknown PET model'):
        ens.EnsembleStatics(10, 2000, 2000, None, None, None, None, None, None, None, 1, np.ones(10), np.ones((1, 5)),
                            np.ones(10), None, None, None, None, pet=name, latitude=np.zeros(10), routing=False)


def _single(rng, shape, nan=True):
    """float64 values that are exactly single precision, with NaN."""
    a = rng.normal(10.0, 5.0, shape).astype(np.float32).astype(np.float64)
    if nan:
        a[rng.random(shape) < 0.05] = np.nan
    return a


@pytest.mark.parametrize("pet", ['hs', 'thornthwaite', 'none'])
def test_lossless_float32_converts_every_pet_models_fields(pet):
    from xanthos_b200 import ensemble as ens
    rng = np.random.default_rng(3)
    member = {k: _single(rng, (7, 24)) for k in ens.forcing_fields(pet)}
    member['tmin'] = rng.normal(0.0, 1.0, (7, 24))                 # not representable: stays float64
    member['extra'] = _single(rng, (7, 24))                        # not a forcing key: left alone
    out = ens.lossless_float32(member, pin=False)
    assert set(out) == set(member)
    for k in ens.forcing_fields(pet):
        if k == 'tmin':
            assert out[k] is member[k]
        else:
            assert out[k].dtype == np.float32
            assert np.array_equal(out[k].astype(np.float64), member[k], equal_nan=True)
    assert out['extra'] is member['extra']


def test_lossless_float32_keeps_a_shared_array_shared():
    from xanthos_b200 import ensemble as ens
    rng = np.random.default_rng(4)
    member = {k: _single(rng, (5, 12)) for k in ('hs_tas', 'hs_tmax', 'hs_tmin', 'precip')}
    member['tmin'] = member['hs_tmin']                             # TempMinFile and hs_tmin: one file
    out = ens.lossless_float32(member, pin=False)
    assert out['tmin'] is out['hs_tmin'] and out['tmin'].dtype == np.float32
    assert len({id(v) for v in out.values()}) == 4
    # a shared array that is not representable stays the one float64 array
    member['hs_tmin'] = member['tmin'] = rng.normal(0.0, 1.0, (5, 12))
    out = ens.lossless_float32(member, pin=False)
    assert out['tmin'] is out['hs_tmin'] is member['tmin']
