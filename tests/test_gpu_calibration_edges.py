"""
GPU tests of the calibration objective (`xan_abcd_kge_batch`) at the edges of its input, in both of its layouts
(block per (candidate, basin) and population: lane = candidate), against oracle/calibrate.py and oracle/abcd.py:
constant series, whose KGE correlation is NaN; candidate counts around the layout switch and up to the maximum;
the shortest spin-up; repeated basins; basins smaller than a chunk; the division fallback for divisors with an
all-ones significand; bit-exact runs where the recurrence has no transcendental; and what the differential-evolution
drivers report for a basin whose forcing is missing everywhere.
"""

import numpy as np
import pytest

from util import max_rel, bitwise_equal

pytestmark = pytest.mark.gpu
RTOL = 1e-9
M, SPIN = 48, 36
LAYOUTS = ('block', 'population')
UNITS = [(True, 'km3_per_mth'), (False, 'mm_per_mth')]
UNIT_IDS = ['km3-snow', 'mm-nosnow']

# Parameters whose divisor has an all-ones significand, so that the kernels take the plain division instead of the
# reciprocal form (significand_all_ones, csrc/abcd.cu): a * 2 = 2 - 2**-52 and d + 1 = 2 - 2**-52.  The third divisor,
# b = pars[1] * 1000, cannot be made one: the only all-ones value of a binade is 2**(k+1) - 2**(k-52), and no double
# x in (1e-4, 8) has fl(x * 1000) equal to it.
ODD_A = np.nextafter(1.0, 0.0)
ODD_D = 1.0 - 2.0 ** -52


def _all_ones(x):
    return (np.float64(x).view(np.int64) & ((1 << 52) - 1)) == (1 << 52) - 1


@pytest.fixture(scope='module')
def world():
    from xanthos_b200 import synthetic
    w = synthetic.make_world(30, 60, 700, 9, seed=61)
    f = synthetic.abcd_inputs(w, M, seed=9)
    f['tmin'] = np.nan_to_num(f['tmin'])
    return w, f


def _pars(rng, nb, npar, snow):
    hi = (0.9999, 7.9999, 0.9999, 0.9999, 0.9999)
    p = np.stack([rng.uniform(1e-4, h, (nb, npar)) for h in hi], axis=2)
    return p if snow else p[:, :, :4]


def _months(f, m):
    return {k: np.ascontiguousarray(f[k][:, :m]) for k in ('precip', 'pet', 'tmin')}


def _evaluator(f, basin_ids, area, snow, unit, m=M, spin=SPIN):
    from xanthos_b200.calibrate import calibrate_abcd as cal
    return cal.BasinEvaluator(basin_ids, area, f['precip'], f['pet'], f['tmin'] if snow else None, m, spin, unit)


def _evaluate(monkeypatch, layout, ev, bnums, pars, obs):
    if layout is None:
        monkeypatch.delenv('XANTHOS_KGE_LAYOUT', raising=False)
    else:
        monkeypatch.setenv('XANTHOS_KGE_LAYOUT', layout)
    return ev.evaluate(np.asarray(bnums), pars, obs, want_series=True)


def _oracle_series(f, basin_ids, area, b, par, snow, unit, m=M, spin=SPIN):
    from oracle import calibrate as ocal
    idx = np.where(basin_ids == b)[0]
    return ocal.basin_series(par, f['pet'][idx], f['precip'][idx], f['tmin'][idx] if snow else None, m, spin, unit,
                             area[idx])


def _check_oracle(results, f, basin_ids, area, bnums, pars, obs, snow, unit, slots, cands, m=M, spin=SPIN):
    """Series and distances of every (ed, series) in `results` against the oracle, for the given slots and candidates;
    the NaN pattern of the distances must agree exactly."""
    from oracle import calibrate as ocal
    for i in slots:
        for p in cands:
            want_s = _oracle_series(f, basin_ids, area, bnums[i], pars[i, p], snow, unit, m, spin)
            with np.errstate(invalid='ignore', divide='ignore'):
                want = ocal.kge_distance(want_s, obs[i])
            for ed, series in results:
                assert max_rel(series[i, p], want_s, floor=1e-12) < RTOL, (bnums[i], p)
                assert max_rel([ed[i, p]], [want]) < RTOL, (bnums[i], p, ed[i, p], want)


# ---- 1. degenerate series --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
@pytest.mark.parametrize("layout", LAYOUTS)
def test_degenerate_series_match_the_oracle(world, layout, snow, unit, monkeypatch):
    """A constant modelled or observed series has no correlation: np.corrcoef gives NaN and so does the distance.
    DE counts NaN as +inf, so a finite value here (r clipped to -1) would make such a basin look converged."""
    w, f = world
    A, B, Z, D, E = 2, 3, 4, 5, 6               # basins of cases (a) .. (e)
    f = dict(f, precip=f['precip'].copy())
    f['precip'][w.basin_ids == A] = np.nan      # (a): every cell of the basin without forcing, modelled series == 0
    nb, P = w.n_basins, 5
    rng = np.random.default_rng(11)
    pars = _pars(rng, nb, P, snow)
    bnums = np.arange(1, nb + 1)
    obs = rng.uniform(0.5, 2.0, (nb, M))
    obs[B - 1] = 1.0                            # (b)
    obs[Z - 1] = 0.0                            # (c): a dry gauge
    obs[D - 1, 17] = np.nan                     # (d)
    # (e): half the oracle series of candidate 0 - correlation 1 up to rounding, relvar = bias = 2 exactly
    obs[E - 1] = 0.5 * _oracle_series(f, w.basin_ids, w.area, E, pars[E - 1, 0], snow, unit)
    ev = _evaluator(f, w.basin_ids, w.area, snow, unit)
    ed, series = _evaluate(monkeypatch, layout, ev, bnums, pars, obs)
    assert (series[A - 1].view(np.int64) == 0).all()             # +0.0 bit for bit: nansum over NaN cells
    assert np.isnan(ed[[A - 1, B - 1, Z - 1, D - 1]]).all(), ed
    assert abs(ed[E - 1, 0] - np.sqrt(2.0)) < RTOL * np.sqrt(2.0), ed[E - 1, 0]
    _check_oracle([(ed, series)], f, w.basin_ids, w.area, bnums, pars, obs, snow, unit, range(nb), range(P))


def test_kge_distance_device_of_degenerate_series():
    """The torch distance of the streamflow objective (no clip) gives the oracle's NaN for cases (a) .. (c)."""
    import torch
    from xanthos_b200.calibrate import calibrate_abcd as cal
    from oracle import calibrate as ocal
    rng = np.random.default_rng(12)
    x, y = rng.uniform(0.5, 2.0, (2, M))
    mod = np.stack([np.zeros(M), x, x, x])[:, None, :]          # [4 basins, 1 candidate, M]
    obs = np.stack([y, np.ones(M), np.zeros(M), y])
    got = cal.kge_distance_device(torch.from_numpy(mod).cuda(), torch.from_numpy(obs).cuda()).cpu().numpy()
    with np.errstate(invalid='ignore', divide='ignore'):
        want = np.array([[ocal.kge_distance(mod[i, 0], obs[i])] for i in range(4)])
    assert np.isnan(got[:3]).all() and np.isfinite(got[3]).all(), got
    assert max_rel(got, want) < RTOL


# ---- 2. shape edges --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("npar", [1, 15, 16, 31, 32, 33, 512])
@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
def test_candidate_counts(world, npar, snow, unit, monkeypatch):
    """Around the switch of layouts (16 candidates), around a group of 32 lanes, and the maximum of 512 (the re-init
    kernel of the population layout then asks for 12 x 512 x 8 B = 48 KB of shared memory)."""
    w, f = world
    nb = w.n_basins
    rng = np.random.default_rng(13 + npar)
    pars = _pars(rng, nb, npar, snow)
    obs = rng.uniform(0.5, 2.0, (nb, M))
    bnums = np.arange(1, nb + 1)
    ev = _evaluator(f, w.basin_ids, w.area, snow, unit)
    ed_b, s_b = _evaluate(monkeypatch, 'block', ev, bnums, pars, obs)
    ed_p, s_p = _evaluate(monkeypatch, 'population', ev, bnums, pars, obs)
    # The layouts add the nanmean of the re-initialisation over the cells in different orders, so the initial state
    # differs in the last bit or two.  For a candidate with a near 1 (a = 0.99985 is among the 9 x 512) the cancellation
    # in awet = w - y amplifies one ulp of the initial state to 5e-13 of the series (measured with the oracle), hence
    # 1e-11 here where test_gpu_model.py's 40 candidates hold 1e-12.
    assert max_rel(s_p, s_b, floor=1e-12) < 1e-11 and max_rel(ed_p, ed_b, floor=1e-12) < 1e-11
    ed_d, s_d = _evaluate(monkeypatch, None, ev, bnums, pars, obs)     # default: block below 16 candidates
    want_ed, want_s = (ed_b, s_b) if npar < 16 else (ed_p, s_p)
    assert bitwise_equal(ed_d, want_ed) and bitwise_equal(s_d, want_s)
    cands = sorted({0, 31, 32, npar // 2, npar - 1} & set(range(npar)))
    _check_oracle([(ed_b, s_b), (ed_p, s_p)], f, w.basin_ids, w.area, bnums, pars, obs, snow, unit, (0, 4, nb - 1),
                  cands)


def test_population_layout_refuses_513_candidates(world, monkeypatch):
    from xanthos_b200 import _cuda as C
    w, f = world
    nb = w.n_basins
    rng = np.random.default_rng(14)
    pars, obs = _pars(rng, nb, 513, True), rng.uniform(0.5, 2.0, (nb, M))
    ev = _evaluator(f, w.basin_ids, w.area, True, 'km3_per_mth')
    for layout in ('population', None):
        with pytest.raises(C.ValidationException):
            _evaluate(monkeypatch, layout, ev, np.arange(1, nb + 1), pars, obs)


@pytest.mark.parametrize("spin", [25, 37])
@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
def test_shortest_and_longest_spinup(world, spin, snow, unit, monkeypatch):
    """37 months (not a multiple of 4 or 12); spin-up 25 puts the three Decembers on months 0, 12 and 24, spin-up 37
    spins up over the whole forcing.  The runoff kernels (abcd_execute) are run at the same edge."""
    from xanthos_b200.runoff import abcd
    from oracle import abcd as oabcd
    w, f0 = world
    m = 37
    f = _months(f0, m)
    nb, P = w.n_basins, 20
    rng = np.random.default_rng(15)
    pars = _pars(rng, nb, P, snow)
    obs = rng.uniform(0.5, 2.0, (nb, m))
    bnums = np.arange(1, nb + 1)
    ev = _evaluator(f, w.basin_ids, w.area, snow, unit, m, spin)
    res = [_evaluate(monkeypatch, layout, ev, bnums, pars, obs) for layout in LAYOUTS]
    assert max_rel(res[1][1], res[0][1], floor=1e-12) < 1e-12 and max_rel(res[1][0], res[0][0], floor=1e-12) < 1e-11
    _check_oracle(res, f, w.basin_ids, w.area, bnums, pars, obs, snow, unit, (0, 4, nb - 1), (0, P - 1), m, spin)
    tmin = f['tmin'] if snow else None
    got = abcd.abcd_execute(nb, w.basin_ids, f['pet'], f['precip'], tmin, f0['pars'], m, spin, -1)
    want = oabcd.abcd_execute(nb, w.basin_ids, f['pet'], f['precip'], tmin, f0['pars'], m, spin)
    for k, g, x in zip(('aet', 'q', 'sav'), got[1:], want[1:]):
        assert max_rel(g, x, floor=1e-6) < RTOL, k


@pytest.mark.parametrize("layout", LAYOUTS)
def test_spinup_out_of_range_is_refused(world, layout, monkeypatch):
    """Spin-up 24: the reference fails indexing month -25 (IndexError); spin-up beyond the forcing is refused."""
    from xanthos_b200 import _cuda as C
    w, f0 = world
    m = 37
    f = _months(f0, m)
    nb = w.n_basins
    rng = np.random.default_rng(16)
    pars, obs = _pars(rng, nb, 3, True), rng.uniform(0.5, 2.0, (nb, m))
    bnums = np.arange(1, nb + 1)
    with pytest.raises(IndexError):
        _evaluate(monkeypatch, layout, _evaluator(f, w.basin_ids, w.area, True, 'km3_per_mth', m, 24), bnums, pars, obs)
    with pytest.raises(C.ValidationException):
        _evaluate(monkeypatch, layout, _evaluator(f, w.basin_ids, w.area, True, 'km3_per_mth', m, m + 1), bnums, pars,
                  obs)


@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
@pytest.mark.parametrize("layout", LAYOUTS)
def test_basin_listed_twice(world, layout, snow, unit, monkeypatch):
    w, f = world
    nb, P = w.n_basins, 20
    rng = np.random.default_rng(17)
    pars = _pars(rng, nb, P, snow)
    obs = rng.uniform(0.5, 2.0, (nb, M))
    ev = _evaluator(f, w.basin_ids, w.area, snow, unit)
    ed, series = _evaluate(monkeypatch, layout, ev, np.arange(1, nb + 1), pars, obs)
    sub = np.array([5, 2, 5, 7])
    ed_s, series_s = _evaluate(monkeypatch, layout, ev, sub, pars[sub - 1], obs[sub - 1])
    assert bitwise_equal(ed_s[0], ed_s[2]) and bitwise_equal(series_s[0], series_s[2])
    assert bitwise_equal(ed_s, ed[sub - 1]) and bitwise_equal(series_s, series[sub - 1])


@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
def test_small_basins_and_chunk_padding(world, snow, unit, monkeypatch):
    """Basins of 1 .. 5 cells (fewer than the 4-cell chunk of the population layout, or one more), and basins whose
    chunk count leaves 0, 1, 2 and 3 padding chunks in the last 4-chunk block."""
    w, f = world
    sizes = (1, 2, 3, 4, 5, 6, 9, 12, 16)
    perm = np.random.default_rng(18).permutation(w.ncell)
    ids = np.full(w.ncell, len(sizes) + 1)                    # the remaining cells form one big basin
    cut = np.cumsum((0,) + sizes)
    for k in range(len(sizes)):
        ids[perm[cut[k]:cut[k + 1]]] = k + 1
    n_cells = np.bincount(ids)[1:]
    pad = (-(-n_cells // 4)) % 4
    assert {1, 2, 3, 4, 5} <= set(n_cells.tolist()) and {0, 1, 2, 3} <= set(pad.tolist()), (n_cells, pad)
    nb, P = len(n_cells), 40
    rng = np.random.default_rng(19)
    pars = _pars(rng, nb, P, snow)
    obs = rng.uniform(0.5, 2.0, (nb, M))
    bnums = np.arange(1, nb + 1)
    ev = _evaluator(f, ids, w.area, snow, unit)
    res = [_evaluate(monkeypatch, layout, ev, bnums, pars, obs) for layout in LAYOUTS]
    assert max_rel(res[1][1], res[0][1], floor=1e-12) < 1e-12 and max_rel(res[1][0], res[0][0], floor=1e-12) < 1e-11
    _check_oracle(res, f, ids, w.area, bnums, pars, obs, snow, unit, range(nb), (0, 31, 32, P - 1))


# ---- 3. division fallback --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
@pytest.mark.parametrize("layout", LAYOUTS)
def test_division_fallback_of_the_objective(world, layout, snow, unit, monkeypatch):
    """Two candidates of one 32-lane group need the plain division; in the population layout they send the whole
    group down that path.  They match the oracle, and the other 30 are bit for bit what a call without them gives."""
    assert _all_ones(ODD_A * 2) and _all_ones(ODD_D + 1)
    w, f = world
    nb, P, odd = w.n_basins, 32, (5, 20)
    rng = np.random.default_rng(20)
    pars = _pars(rng, nb, P, snow)
    pars[:, odd[0], 0] = ODD_A
    # With a = 1 - 2**-53 and w < b, awet = w - y is a difference of equal numbers: the runoff is rounding residue, and
    # one ulp of PET in the oracle moves the late months of the series by up to 18 %.  b = 20 mm keeps w > b in most
    # months; the same ulp then moves the series by 2e-15.  (The plain division itself is checked bit for bit below.)
    pars[:, odd[0], 1] = 0.02
    pars[:, odd[1], 3] = ODD_D
    obs = rng.uniform(0.5, 2.0, (nb, M))
    bnums = np.arange(1, nb + 1)
    ev = _evaluator(f, w.basin_ids, w.area, snow, unit)
    ed, series = _evaluate(monkeypatch, layout, ev, bnums, pars, obs)
    keep = [p for p in range(P) if p not in odd]
    ed_f, series_f = _evaluate(monkeypatch, layout, ev, bnums, pars[:, keep], obs)
    assert bitwise_equal(ed[:, keep], ed_f) and bitwise_equal(series[:, keep], series_f)
    _check_oracle([(ed, series)], f, w.basin_ids, w.area, bnums, pars, obs, snow, unit, range(nb), odd)


@pytest.mark.parametrize("snow", [True, False])
def test_division_fallback_of_the_runoff_kernels(world, snow):
    from xanthos_b200.runoff import abcd
    from oracle import abcd as oabcd
    w, f = world
    pars = f['pars'].copy()
    pars[1, 0] = ODD_A
    pars[2, 3] = ODD_D
    tmin = f['tmin'] if snow else None
    got = abcd.abcd_execute(w.n_basins, w.basin_ids, f['pet'], f['precip'], tmin, pars, M, SPIN, -1)
    want = oabcd.abcd_execute(w.n_basins, w.basin_ids, f['pet'], f['precip'], tmin, pars, M, SPIN)
    for k, g, x in zip(('aet', 'q', 'sav'), got[1:], want[1:]):
        assert max_rel(g, x, floor=1e-6) < RTOL, k


# ---- 4. bit for bit with zero PET ------------------------------------------------------------------------------------
# With PET == 0, exp(-0 / b) is exactly 1 in CUDA and numpy alike; what is left of the recurrence is + - * / and sqrt,
# all correctly rounded (FMA contraction is off, and the reciprocal form of the division claims correct rounding).
# With one cell per basin the nanmean of the re-initialisation and the nansum of the basin series add one value to
# zeros.  So any difference, even of one bit, comes from an operation that is not the reference's.

@pytest.mark.parametrize("snow", [True, False])
def test_runoff_is_bitwise_the_oracle_with_zero_pet(world, snow):
    from xanthos_b200.runoff import abcd
    from oracle import abcd as oabcd
    w, f = world
    n = w.ncell
    ids = np.arange(1, n + 1)
    pars = _pars(np.random.default_rng(21), n, 1, True)[:, 0, :]
    pars[1, 0] = ODD_A                                        # two cells on the plain division
    pars[2, 3] = ODD_D
    pet = np.zeros_like(f['pet'])
    tmin = f['tmin'] if snow else None
    got = abcd.abcd_execute(n, ids, pet, f['precip'], tmin, pars, M, SPIN, -1)
    want = oabcd.abcd_execute(n, ids, pet, f['precip'], tmin, pars, M, SPIN)
    for k, g, x in zip(('aet', 'q', 'sav'), got[1:], want[1:]):
        assert bitwise_equal(g, x), (k, max_rel(g, x, floor=1e-6))


@pytest.mark.parametrize("snow,unit", UNITS, ids=UNIT_IDS)
def test_objective_series_is_bitwise_the_oracle_with_zero_pet(world, snow, unit, monkeypatch):
    w, f = world
    f = dict(f, pet=np.zeros_like(f['pet']))
    nan_cell = np.nonzero(np.isnan(f['precip']).any(axis=1))[0][:1]      # a cell with a missing month
    cells = np.concatenate([np.setdiff1d(np.arange(24), nan_cell)[:23], nan_cell])
    ids = np.zeros(w.ncell, dtype=int)                        # the other cells are in no basin
    ids[cells] = np.arange(1, len(cells) + 1)
    nb, P = len(cells), 20
    rng = np.random.default_rng(22)
    pars = _pars(rng, nb, P, snow)
    pars[:, 3, 0] = ODD_A                                     # the first 32-lane group takes the plain division
    pars[:, 7, 3] = ODD_D
    obs = rng.uniform(0.5, 2.0, (nb, M))
    bnums = np.arange(1, nb + 1)
    ev = _evaluator(f, ids, w.area, snow, unit)
    res = [_evaluate(monkeypatch, layout, ev, bnums, pars, obs) for layout in LAYOUTS]
    for i in range(nb):
        for p in range(P):
            want = _oracle_series(f, ids, w.area, i + 1, pars[i, p], snow, unit)
            for layout, (_, series) in zip(LAYOUTS, res):
                assert bitwise_equal(series[i, p], want), (layout, i + 1, p, max_rel(series[i, p], want, floor=1e-12))


# ---- 5. what the drivers report --------------------------------------------------------------------------------------

@pytest.mark.parametrize("popsize", [2, 15])               # 10 candidates: block layout; 75: population layout
@pytest.mark.parametrize("driver", ['device', 'host'])
def test_driver_keeps_a_basin_without_forcing_unconverged(world, driver, popsize, monkeypatch):
    """Every candidate of a basin whose forcing is missing everywhere scores NaN, counted as +inf: the basin runs to
    maxiter and reports KGE = -inf instead of converging at initialisation on a finite distance."""
    from xanthos_b200.calibrate import calibrate_abcd as cal
    monkeypatch.delenv('XANTHOS_KGE_LAYOUT', raising=False)
    w, f = world
    dead = 3
    precip = f['precip'].copy()
    precip[w.basin_ids == dead] = np.nan
    bnums = np.arange(1, w.n_basins + 1)
    vals = np.random.default_rng(23).uniform(0.5, 2.0, (w.n_basins, M))
    obs = np.concatenate([np.column_stack([np.full(M, b), vals[b - 1]]) for b in bnums])
    _, kge, info = cal.calibrate_basins(bnums, w.basin_ids, w.area, precip, f['pet'], obs, f['tmin'], M, SPIN,
                                        'km3_per_mth', popsize=popsize, maxiter=3, seed=5, driver=driver)
    i = dead - 1
    assert kge[i] == -np.inf and info['nit'][i] == 3 and info['fun'][i] == np.inf, (kge[i], info['nit'][i])
    assert np.isfinite(np.delete(kge, i)).all(), kge
