"""
CPU tests: the numpy oracle against (a) the committed golden fixtures that were
produced by running the reference, (b) the reference's own known-answer test
(xanthos/test/test_thornthwaite.py) and (c) the live reference when
/root/reference is present (build container only).
"""

import numpy as np
import pytest

from oracle import pet as opet, mrtm as omrtm, abcd as oabcd
from oracle import ref_loader
from oracle.validate_against_reference import (run_oracle, oracle_calibration, build_case, run_reference, compare,
                                               run_oracle_stepwise, build_stepwise_case, run_reference_stepwise)
from oracle.calendar_utils import set_month_arrays
from util import load_golden, bitwise_equal


@pytest.mark.parametrize("name", ["case_a", "case_b"])
def test_oracle_matches_golden_bitwise(name):
    case, ref = load_golden(name)
    out = run_oracle(case)
    for k, v in out.items():
        assert bitwise_equal(v, ref[k]), k
    ed = oracle_calibration(case, ref)
    assert np.max(np.abs(ed - ref['cal_ed']) / np.abs(ref['cal_ed'])) < 1e-12


def test_stepwise_oracle_matches_golden_bitwise():
    """Hargreaves PET + GWAM runoff with its spin-up pass (tests/golden/case_c.npz, produced by the reference)."""
    case, ref = load_golden("case_c")
    out = run_oracle_stepwise(case)
    assert set(out) == set(ref)
    for k, v in out.items():
        assert bitwise_equal(v, ref[k]), k


def test_postproc_oracle_matches_golden_bitwise():
    """Drought statistics, Aggregation_Map and the accessible-water chain (tests/golden/case_d.npz, produced by the
    reference's own functions)."""
    from oracle.validate_against_reference import run_oracle_postproc
    case, ref = load_golden("case_d")
    out = run_oracle_postproc(case)
    assert set(out) == set(ref)
    for k, v in out.items():
        assert bitwise_equal(v, ref[k]), k
    assert np.isnan(ref['thr12']).any() and (ref['dur12'].max() > 12)      # the edge cases are really in the fixture


def test_upstream_fast_equals_loop():
    case, ref = load_golden("case_a")
    a = omrtm.upstream_fast(case['coords'], ref['dsid'], case['nrow'], case['ncol'])
    assert np.array_equal(a, ref['upid'])


def test_thornthwaite_known_answer():
    """xanthos/test/test_thornthwaite.py:12-37, restated for the oracle."""
    days = [31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31]
    eq = opet.daylight_hours(days, np.array([0.0]))
    npole = opet.daylight_hours(days, np.array([np.pi / 2]))
    spole = opet.daylight_hours(days, np.array([-np.pi / 2]))
    assert np.all(eq == 12)
    assert np.any(npole[0] == 0.0) and np.any(npole[0] == 24.0)
    assert np.all(24 - npole == spole)
    lat = np.array([0.698132])
    tas1 = np.array([[2, 5, 6, 8, 10, 12, 15, 12, 10, 8, 6, 5]], dtype=float)
    tas2 = -np.ones((1, 12))
    want = np.array([[9.7, 22.9, 33.7, 47.6, 66.0, 78.8, 98.5, 74.4, 54.8, 40.9, 27.1, 22.3]])
    assert np.all(np.round(opet.thornthwaite_pet(tas1, lat, 1999, 1999), 1) == want)
    assert np.all(opet.thornthwaite_pet(tas2, lat, 1999, 1999) == 0)


def test_abcd_spinup_too_short_raises():
    case, _ = load_golden("case_a")
    with pytest.raises(IndexError):
        oabcd.abcd_execute(case['n_basins'], case['basin_ids'], case['abcd_pet'], case['precip'],
                           np.nan_to_num(case['tmin']), case['abcd_pars'], case['nmonths'], 24)


def test_kge_distance_of_a_constant_series_is_nan():
    """The KGE correlation of the reference is np.corrcoef, which is NaN when either series is constant (zero
    variance) and keeps that NaN through its np.clip: the distance is NaN, not a finite value from r = -1."""
    from oracle.calibrate import kge_distance
    rng = np.random.default_rng(0)
    varying = rng.uniform(0.5, 2.0, 48)
    cases = [(np.zeros(48), varying),          # modelled == 0: every cell of the basin has missing forcing
             (varying, np.ones(48)),           # observed == 1
             (varying, np.zeros(48))]          # observed == 0: a dry gauge
    with np.errstate(invalid='ignore', divide='ignore'):
        for mod, obs in cases:
            assert np.isnan(np.corrcoef(obs, mod)[1, 0])
            assert np.isnan(kge_distance(mod, obs))
        # a correlation of 1 is kept (clipped if it rounds above 1): relvar = bias = 2 exactly
        assert kge_distance(varying, 0.5 * varying) == pytest.approx(np.sqrt(2.0), rel=1e-12)


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
def test_oracle_matches_live_reference():
    case = build_case(nrow=20, ncol=40, ncell=180, n_basins=5, seed=77, start_yr=2003, end_yr=2005,
                      spinup=30, routing_spinup=2)
    r = run_reference(case)
    o = run_oracle(case)
    for k, (bit, rel, same_nan) in compare(r, o, verbose=False).items():
        assert bit, (k, rel)
    sc = build_stepwise_case(nrow=20, ncol=40, ncell=180, n_basins=5, seed=78, start_yr=2003, end_yr=2004, spinup=9)
    r, o = run_reference_stepwise(sc), run_oracle_stepwise(sc)
    for k in r:
        assert bitwise_equal(r[k], o[k]), k


def test_csr_operator_equals_gather_bitwise():
    """oracle.mrtm.csr_rows (scipy CSR, what the reference multiplies with) and the numpy gather give the same
    routing bit for bit, clamp events included - the CSR form is what the full-size GPU parity tests use."""
    from xanthos_b200 import synthetic
    w = synthetic.make_world(30, 60, 700, 9, seed=61)
    dsid = omrtm.downstream(w.coords, w.flow_dir, w.nrow, w.ncol)
    upid = omrtm.upstream_fast(w.coords, dsid, w.nrow, w.ncol)
    q = synthetic.runoff_input(w, 5, seed=2)
    nd = set_month_arrays(12, 1999, 1999)[:5, 2]
    a = omrtm.route(q, w.flow_dist, w.velocity, w.area, nd, 10800, omrtm.gather_rows(upid), 2)
    b = omrtm.route(q, w.flow_dist, w.velocity, w.area, nd, 10800, omrtm.csr_rows(upid), 2)
    for x, y in zip(a, b):
        assert bitwise_equal(x, y)
    assert ((w.velocity / w.flow_dist) * 10800 > 1).any()          # the world has cells that empty (clamp branch)


@pytest.mark.parametrize("seed,prob", [(12345, 0), (99, 3), (2 ** 40 + 7, 1)])
def test_de_oracle_is_bitwise_scipy_deferred(seed, prob):
    """SURVEY section 8 row f4 / parity of the third-party solver: scipy's own DifferentialEvolutionSolver
    (best1bin, updating='deferred'), fed the Philox stream of the kernels in its own consumption order, produces the
    trial vectors, the selection and the convergence decision of oracle.de bit for bit, out-of-bounds redraws included."""
    from oracle import de
    target = np.array([0.1, -0.2, 0.3, 0.0, -0.4])

    def f(p):
        x = np.asarray(p)
        return float(np.sum((x - target) ** 2) + 0.1 * np.sum(np.cos(7 * x)))
    gens = de.replay_against_scipy(f, 15, S=25, D=5, prob=prob, seed=seed)
    assert len(gens) == 15
    for g in gens:
        assert g['trial_equal'] and g['pop_equal'] and g['energy_equal'] and g['converged_equal'] and g['best_at_row0'], g
    assert sum(g['n_oob'] for g in gens) > 20            # the out-of-bounds branch was exercised
    # a 4-dimensional problem (the no-snow parameter set) with the reference's population (15 x D)
    gens = de.replay_against_scipy(lambda p: float(np.sum(np.asarray(p) ** 2)), 6, S=60, D=4, prob=0, seed=seed)
    assert all(g['trial_equal'] and g['pop_equal'] and g['energy_equal'] for g in gens)


def test_de_oracle_latin_hypercube():
    from oracle import de
    S, D = 50, 5
    p = de.lhs_init(3, S, D, 777)
    assert (p >= 0).all() and (p < 1).all()
    assert (np.sort(np.floor(p * S).astype(int), axis=1) == np.arange(S)[None, :, None]).all()   # every stratum once


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
def test_reference_streamflow_branch_has_no_usable_behaviour():
    """Why the streamflow calibration target (`set_calibrate = 1`) is built to its INTENDED semantics and not to the
    reference's (oracle/calibrate.py docstring): the live reference's own `basin_runoff` / `objective_kge`
    (calibrate_abcd.py:164-213), run here on a small world with a real router, (1) put only the first n_b values of the
    basin's [months, n_b] runoff at FLAT indices of the global [ncell, months] array - rows near the top of the grid, not
    the basin's cells -, (2) hand the router's whole [ncell, months] Avg_ChFlow back as the "modelled series", and
    (3) evaluate to NaN."""
    import numpy as np
    from types import SimpleNamespace
    from xanthos_b200 import synthetic
    from oracle.calendar_utils import set_month_arrays
    ref = ref_loader.load()
    w = synthetic.make_world(24, 48, 320, 5, seed=44)
    m = 36
    ab = synthetic.abcd_inputs(w, m, seed=9)
    tmin = np.nan_to_num(ab['tmin'])
    nd = set_month_arrays(m, 2001, 2003)[:, 2]
    rows = omrtm.csr_rows(omrtm.upstream_fast(w.coords, omrtm.downstream(w.coords, w.flow_dir, w.nrow, w.ncol), w.nrow, w.ncol))
    seen = {}

    def router(rsim):          # stands for Components.calculate_routing (components.py:249-296): returns Avg_ChFlow
        seen['rsim'] = np.array(rsim)
        return omrtm.route(rsim, w.flow_dist, w.velocity, w.area, nd, 10800, rows, 6)[1]
    idx = np.where(w.basin_ids == 3)
    n_b = len(idx[0])
    args = (ab['pet'][idx], ab['precip'][idx], tmin[idx], m, m, 'm3_per_sec', w.area[idx])
    mod = ref.cal.basin_runoff(ab['pars'][2], 1, *args, idx, ab['pet'].shape, router)
    assert np.shape(mod) == ab['pet'].shape                                   # (2): not a series of the basin
    flat = np.nonzero(seen['rsim'].ravel())[0]
    assert len(flat) <= n_b and flat.max() <= idx[0].max()                     # (1): n_b values at flat indices = cell ids
    assert not np.array_equal(np.unique(flat // m), idx[0])                    # ... which are not the basin's rows
    with np.errstate(all='ignore'):
        ed = ref.cal.objective_kge(ab['pars'][2], ref.cal.basin_runoff, 1, *args, np.linspace(1.0, 2.0, m), idx,
                                   ab['pet'].shape, router)
    assert np.isnan(ed)                                                       # (3)
