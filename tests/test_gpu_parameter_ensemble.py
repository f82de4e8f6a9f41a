"""Parameter ensembles: xan_abcd_run_sets is S calls of xan_abcd_run bit for bit, and run_parameter_ensemble gives every
set what the plug-in calls give on that table alone (PET -> abcd_execute(..., pars_k, ...) -> mrtm.route), uploads the
forcing once, applies the output options over the sets and refuses what cannot run."""

import ctypes
from types import SimpleNamespace

import numpy as np
import pytest

from util import bitwise_equal, max_rel

pytestmark = pytest.mark.gpu

SY, EY, M = 1991, 1993, 36
ROUTED_VARS = ('aet', 'q', 'soilmoisture', 'chstorage', 'avgchflow')
UNROUTED_VARS = ROUTED_VARS[:3]


@pytest.fixture(scope='module')
def world():
    from xanthos_b200 import synthetic, ensemble as ens
    from xanthos_b200.routing import mrtm
    from oracle.calendar_utils import set_month_arrays
    w = synthetic.make_world(24, 48, 700, 6, seed=31)
    s = w.settings()
    um = mrtm.upstream_genmatrix(mrtm.upstream(w.coords, mrtm.downstream(w.coords, w.flow_dir, s), s))
    nd = set_month_arrays(M, SY, EY)[:, 2]
    ab = synthetic.abcd_inputs(w, M, seed=20, with_pet=True)            # precip keeps its NaN, as the loader does
    hs = synthetic.hs_inputs(w, SY, EY, seed=40)                        # NaN kept in hs_*
    assert np.isnan(ab['precip']).any() and np.isnan(hs['hs_tas']).any()
    pm = synthetic.pm_inputs(w, SY, EY, nlcs=8, seed=10)
    pm_statics = dict(pm_tables={k: v for k, v in pm.items() if k not in ens.PM_FORCING + ('lct_load', 'tairprev_load')},
                      lct_load=pm['lct_load'], elev=pm['elev'], water_idx=pm['water_idx'], snow_idx=pm['snow_idx'],
                      lc_years=pm['lc_years'], nlcs=8)
    forcing = {'hs': dict({k: hs[k] for k in ('hs_tas', 'hs_tmax', 'hs_tmin')}, precip=ab['precip'], tmin=ab['tmin']),
               'none': dict(pet=ab['pet'], precip=ab['precip'], tmin=ab['tmin']),
               'pm': dict({k: np.nan_to_num(pm[k]) for k in ens.PM_FORCING}, precip=ab['precip'],
                          tmin=np.nan_to_num(ab['tmin']))}
    return SimpleNamespace(w=w, um=um, nd=nd, pars=ab['pars'], ab=ab, forcing=forcing, pm_statics=pm_statics)


def tables(pars, n, seed=5):
    """n parameter tables: the world's table, then tables scaled per entry by factors in [0.8, 1]."""
    rng = np.random.default_rng(seed)
    out = np.repeat(np.asarray(pars, dtype=np.float64)[None], n, axis=0)
    out[1:] *= rng.uniform(0.8, 1.0, out[1:].shape)
    return out


def statics(wd, pet, routing):
    from xanthos_b200 import ensemble as ens
    w = wd.w
    kw = dict(ncell=w.ncell, start_yr=SY, end_yr=EY, pm_tables=None, lct_load=None, elev=None, water_idx=None,
              snow_idx=None, lc_years=None, nlcs=None, n_basins=w.n_basins, basin_ids=w.basin_ids, abcd_pars=wd.pars,
              area=w.area, flow_dist=None, velocity=None, upstream_matrix=None, ndays=None, dt=10800, runoff_spinup=M,
              routing_spinup=6, pet=pet, latitude=w.coords[:, 2] if pet == 'hs' else None, routing=routing)
    if routing:
        kw.update(flow_dist=w.flow_dist, velocity=w.velocity, upstream_matrix=wd.um, ndays=wd.nd)
    if pet == 'pm':
        kw.update(wd.pm_statics)
    return ens.EnsembleStatics(**kw)


def standalone(wd, pet, pars, routing):
    """Table `pars` through the plug-in calls on the world's forcing of PET model `pet`."""
    from xanthos_b200.pet import hargreaves_samani, penman_monteith as pm_mod
    from xanthos_b200.runoff import abcd
    from xanthos_b200.routing import mrtm
    w, mem = wd.w, wd.forcing[pet]
    if pet == 'hs':
        data = SimpleNamespace(coords=w.coords, hs_tas=mem['hs_tas'], hs_tmax=mem['hs_tmax'], hs_tmin=mem['hs_tmin'])
        p = hargreaves_samani.execute(SimpleNamespace(StartYear=SY), data)
    elif pet == 'pm':
        ps = wd.pm_statics
        data = SimpleNamespace(**{**ps['pm_tables'], 'lct_load': ps['lct_load'], 'elev': ps['elev'], **mem})
        p = pm_mod.run_pmpet(data, w.ncell, 8, SY, EY, ps['water_idx'], ps['snow_idx'], ps['lc_years'])
    else:
        p = mem['pet']
    _, aet, q, sav = abcd.abcd_execute(w.n_basins, w.basin_ids, p, mem['precip'], np.nan_to_num(mem['tmin']), pars,
                                       M, M, -1)
    out = {'aet': aet, 'q': q, 'soilmoisture': sav}
    if routing:
        chs, avg, _ = mrtm.route(wd.um, q, w.flow_dist, w.velocity, w.area, wd.nd, 10800, 6)
        out.update(chstorage=chs, avgchflow=avg)
    return out


def check_sets(wd, res, sets, pet, routing, output_vars):
    w = wd.w
    rows = 2 if routing else 1
    assert res['basin_aggregates'].shape == (len(sets), rows, M, w.n_basins)
    assert res['stats']['members_local'] == len(sets)
    wants = []
    for k, pars in enumerate(sets):
        want = standalone(wd, pet, pars, routing)
        wants.append(want)
        assert 'pet' not in res[k]
        for v in output_vars:
            assert bitwise_equal(res[k][v], want[v]), (k, v)
        for b in range(w.n_basins):
            idx = w.basin_ids == b + 1
            q_b = np.nansum(want['q'][idx] * (w.area[idx] * 1e-6)[:, None], axis=0)
            assert max_rel(res['basin_aggregates'][k, 0, :, b], q_b, floor=1e-12) < 1e-12
            if routing:
                f_b = np.nansum(want['avgchflow'][idx], axis=0)
                assert max_rel(res['basin_aggregates'][k, 1, :, b], f_b, floor=1e-12) < 1e-12
    return wants


# ---- the kernel ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def kernel_inputs(world):
    """Month-major forcing and a plan over all basins but the last: its cells are outside the basin range (NaN), and the
    tables have more rows than the plan (as EnsembleStatics' abcd_pars rows > n_basins)."""
    from xanthos_b200 import _cuda as C
    from xanthos_b200.runoff import abcd
    w, ab = world.w, world.ab
    assert w.ncell % 128 != 0
    nb = w.n_basins - 1
    rows = abcd._basin_rows(nb, w.basin_ids, w.n_basins)
    assert (rows < 0).any() and (rows >= 0).any()
    plan = abcd.basin_plan(rows, nb)
    e, p = C.Field.from_host(ab['pet']), C.Field.from_host(ab['precip'])
    t = C.Field.from_host(np.nan_to_num(ab['tmin']))
    return SimpleNamespace(plan=plan, e=e, p=p, t=t, rows=rows, ncell=w.ncell)


def same_bits(a, b, ncell):
    """Two month-major Fields hold the same bits in the first ncell columns (NaN payloads included)."""
    import torch
    return torch.equal(a.t[:, :ncell].contiguous().view(torch.int64), b.t[:, :ncell].contiguous().view(torch.int64))


def special_tables(world, n):
    """n tables; set 1 has a = 0.9999999999999999 in every row (2a has an all-ones significand: the generic division),
    set 2 a NaN b in the first row."""
    sets = tables(world.pars, n)
    if n > 1:
        sets[1, :, 0] = 0.9999999999999999
        assert (np.asarray(2 * sets[1, 0, 0]).view(np.int64) & ((1 << 52) - 1)) == (1 << 52) - 1
    if n > 2:
        sets[2, 0, 1] = np.nan
    return sets


@pytest.mark.parametrize("snow", [True, False])
@pytest.mark.parametrize("n_sets", [1, 2, 3, 8, 19])
def test_run_sets_equals_single_runs(world, kernel_inputs, n_sets, snow):
    from xanthos_b200 import _cuda as C
    from xanthos_b200.runoff import abcd
    ki = kernel_inputs
    assert C.ABCD_MAX_SETS == 8
    sets = special_tables(world, n_sets)
    t = ki.t if snow else None
    got = abcd.run_device_sets(ki.plan, sets, ki.e, ki.p, t, M, M)
    assert len(got) == n_sets
    for k in range(n_sets):
        want = abcd.run_device(ki.plan, sets[k], ki.e, ki.p, t, M, M)
        for v in ('aet', 'q', 'sav'):
            assert same_bits(got[k][v], want[v], ki.ncell), (k, v)
            x = got[k][v].t[:, :ki.ncell].cpu().numpy()
            assert np.isnan(x[:, ki.rows < 0]).all()
            if k != 2:
                assert not np.isnan(x[:, ki.rows >= 0]).all()
    if n_sets > 2:      # the NaN parameter reaches the cells of its basin
        q2 = got[2]['q'].t[:, :ki.ncell].cpu().numpy()
        assert np.isnan(q2[:, ki.rows == 0]).all()


def test_run_sets_null_outputs(world, kernel_inputs):
    import torch
    from xanthos_b200 import _cuda as C
    from xanthos_b200.runoff import abcd
    ki, S = kernel_inputs, 3
    sets = torch.from_numpy(tables(world.pars, S)).cuda()
    fill = float.fromhex('0x1.5p+7')
    q = [C.Field.empty(ki.ncell, M, ki.e.ld) for _ in range(S)]
    sav = [C.Field.empty(ki.ncell, M, ki.e.ld) for _ in range(S)]
    for f in q + sav:
        f.t.fill_(fill)
    h_q = (ctypes.c_void_p * S)(q[0].t.data_ptr(), None, q[2].t.data_ptr())
    h_sav = (ctypes.c_void_p * S)(*[f.t.data_ptr() for f in sav])
    C.check(C.lib().xan_abcd_run_sets(ki.plan._plan, S, sets.shape[1], C.ptr(ki.e.t), C.ptr(ki.p.t), C.ptr(ki.t.t),
                                      C.ptr(sets), M, M, ki.e.ld, None, h_q, h_sav, C.stream_ptr()))
    assert bool((q[1].t == fill).all())
    for k in range(S):
        want = abcd.run_device(ki.plan, sets[k], ki.e, ki.p, ki.t, M, M)
        assert same_bits(sav[k], want['sav'], ki.ncell), k
        if k != 1:
            assert same_bits(q[k], want['q'], ki.ncell), k
    C.check(C.lib().xan_abcd_run_sets(ki.plan._plan, S, sets.shape[1], C.ptr(ki.e.t), C.ptr(ki.p.t), C.ptr(ki.t.t),
                                      C.ptr(sets), M, M, ki.e.ld, None, None, None, C.stream_ptr()))


def test_run_sets_refusals(world, kernel_inputs):
    import torch
    from xanthos_b200 import _cuda as C
    ki = kernel_inputs
    sets = torch.from_numpy(tables(world.pars, C.ABCD_MAX_SETS + 1)).cuda()
    n_rows = int(sets.shape[1])

    def call(n_sets=2, rows=n_rows, pars=C.ptr(sets), spinup=M, pet=C.ptr(ki.e.t)):
        return C.lib().xan_abcd_run_sets(ki.plan._plan, n_sets, rows, pet, C.ptr(ki.p.t), C.ptr(ki.t.t), pars, M,
                                         spinup, ki.e.ld, None, None, None, C.stream_ptr())
    for kw in (dict(n_sets=0), dict(n_sets=C.ABCD_MAX_SETS + 1), dict(rows=0), dict(pars=None), dict(pet=None),
               dict(rows=world.w.n_basins - 2)):      # the plan maps cells to row n_basins - 2
        with pytest.raises(C.ValidationException):
            C.check(call(**kw))
    assert call(spinup=24) == C.XAN_E_SPINUP
    with pytest.raises(IndexError, match='spin-up'):
        C.check(call(spinup=24))
    C.check(call(n_sets=C.ABCD_MAX_SETS))
    torch.cuda.synchronize()


# ---- the runner ---------------------------------------------------------------------------------------------------
def test_pm_routed_five_sets(world):
    from xanthos_b200 import ensemble as ens
    sets = tables(world.pars, 5)
    res = ens.run_parameter_ensemble(statics(world, 'pm', True), world.forcing['pm'], sets, output_vars=ROUTED_VARS)
    check_sets(world, res, sets, 'pm', True, ROUTED_VARS)


def test_hs_unrouted_nine_sets(world):
    from xanthos_b200 import ensemble as ens
    sets = special_tables(world, 9)
    st = statics(world, 'hs', False)
    res = ens.run_parameter_ensemble(st, world.forcing['hs'], sets, output_vars=UNROUTED_VARS)
    check_sets(world, res, sets, 'hs', False, UNROUTED_VARS)


@pytest.mark.parametrize("routing", [True, False])
def test_given_pet_sets_equal_the_plugin_calls_and_runs_of_one_table(world, routing):
    from xanthos_b200 import ensemble as ens
    sets = tables(world.pars, 5)
    st = statics(world, 'none', routing)
    out_vars = ROUTED_VARS if routing else UNROUTED_VARS
    res = ens.run_parameter_ensemble(st, world.forcing['none'], sets, output_vars=out_vars)
    check_sets(world, res, sets, 'none', routing, out_vars)
    for k in range(len(sets)):       # a set does not depend on its neighbours
        alone = ens.run_parameter_ensemble(st, world.forcing['none'], sets[k:k + 1], output_vars=out_vars)
        for v in out_vars:
            assert bitwise_equal(alone[0][v], res[k][v]), (k, v)
        assert bitwise_equal(alone['basin_aggregates'][0], res['basin_aggregates'][k])


def test_forcing_crosses_the_link_once(world):
    from xanthos_b200 import ensemble as ens
    mem = world.forcing['hs']
    field_bytes = sum({id(a): np.asarray(a).nbytes for a in mem.values()}.values())
    assert field_bytes == 5 * 8 * world.w.ncell * M
    st = statics(world, 'hs', False)
    for n in (1, 6):
        res = ens.run_parameter_ensemble(st, mem, tables(world.pars, n), output_vars=('q',))
        assert res['stats']['h2d_bytes'] == field_bytes, n


def test_four_column_tables_are_tables_without_snow_melt(world):
    from xanthos_b200 import ensemble as ens
    sets = tables(world.pars, 3)
    sets[:, :, 4] = 0.0
    st = statics(world, 'none', False)
    five = ens.run_parameter_ensemble(st, world.forcing['none'], sets, output_vars=UNROUTED_VARS)
    four = ens.run_parameter_ensemble(st, world.forcing['none'], [t[:, :4] for t in sets], output_vars=UNROUTED_VARS)
    for k in range(3):
        for v in UNROUTED_VARS:
            assert bitwise_equal(four[k][v], five[k][v]), (k, v)


def test_output_options_over_the_sets(world):
    """Yearly km3 grids, basin sums, statistics, quantiles and drought of q over the sets: what OutWriter, numpy and
    DroughtStats make of the stand-alone sets' outputs."""
    from xanthos_b200 import ensemble as ens, _cuda as C
    from xanthos_b200.data_writer import out_writer
    from xanthos_b200.diagnostics.time_series import group_sum_device
    from xanthos_b200.drought.drought_stats import DroughtStats
    w = world.w
    sets = tables(world.pars, 5)
    out_vars, levels, years, nper = ('q', 'soilmoisture'), (0.05, 0.5, 0.95), (1992, 1993), 4
    spec = ens.OutputSpec(output_in_year=True, output_unit='km3', group_sums=('basin',), stats=ens.STATS,
                          quantiles=levels, drought=ens.DroughtSpec('q', threshold_years=years, nper=nper))
    res = ens.run_parameter_ensemble(statics(world, 'hs', False), world.forcing['hs'], sets, output_vars=out_vars,
                                     spec=spec)
    n, ny = len(sets), M // 12
    settings = SimpleNamespace(StartYear=SY, threshold_start_year=years[0], threshold_end_year=years[1],
                               threshold_nper=nper)
    stacks, dry = {v: [] for v in out_vars}, 0
    for k in range(n):
        monthly = standalone(world, 'hs', sets[k], False)
        for v in out_vars:
            a = out_writer.agg_to_year(C.remember(np.array(monthly[v]), C.Field.from_host(monthly[v])), 'sum')
            a = np.asarray(a) * (np.asarray(w.area) / 1e6)[:, None]
            assert res[k][v].shape == (w.ncell, ny) and bitwise_equal(res[k][v], a), (k, v)
            stacks[v].append(a)
            if v == 'q':
                basin = group_sum_device(w.basin_ids, C.Field.from_host(a).t).cpu().numpy()
                assert bitwise_equal(res['group_sums']['basin'][k], basin)
        x = np.ascontiguousarray(monthly['q'].T)
        th = DroughtStats.calculate_thresholds(x, settings)
        S_, I_, D_ = DroughtStats.droughtstats(None, x, th)
        assert bitwise_equal(res[k]['drought']['thresholds'], th)
        with np.errstate(invalid='ignore'):
            summ = np.stack([(D_ > 0).sum(0), (D_ == 1).sum(0), D_.max(0), S_.max(0)]).astype(np.float64)
        assert bitwise_equal(res['drought_summary'][k], summ)
        dry = dry + (D_ > 0).astype(np.int32)
    assert np.array_equal(res['ensemble_drought']['members_in_drought'], dry.T)
    assert res['ensemble_drought']['n_members'] == n
    assert res['ensemble_stats']['n_members'] == n and res['ensemble_quantiles']['n_members'] == n
    for v in out_vars:
        x = np.stack(stacks[v])
        with np.errstate(invalid='ignore'):
            ref = {'mean': np.mean(x, axis=0), 'min': np.min(x, axis=0), 'max': np.max(x, axis=0)}
            std = np.std(x, axis=0)
        for st in ref:
            assert bitwise_equal(res['ensemble_stats'][v][st], ref[st]), (v, st)
        ok = ~np.isnan(std)
        np.testing.assert_allclose(res['ensemble_stats'][v]['std'][ok], std[ok], rtol=1e-12,
                                   atol=1e-15 * np.nanmax(np.abs(x)))
        assert bitwise_equal(res['ensemble_quantiles'][v], np.quantile(x, levels, axis=0)), v


def test_refusals(world):
    from xanthos_b200 import ensemble as ens, _cuda as C
    st_r, st_u = statics(world, 'none', True), statics(world, 'none', False)
    mem, sets = world.forcing['none'], tables(world.pars, 2)
    with pytest.raises(C.ValidationException, match="'pet'.*same for every parameter set"):
        ens.run_parameter_ensemble(st_r, mem, sets, output_vars=('q', 'pet'))
    with pytest.raises(C.ValidationException, match='routing'):
        ens.run_parameter_ensemble(st_u, mem, sets, output_vars=('q', 'chstorage'))
    with pytest.raises(C.ValidationException, match='at most 256'):
        ens.run_parameter_ensemble(st_u, mem, tables(world.pars, 257), output_vars=('q',),
                                   spec=ens.OutputSpec(quantiles=(0.5,)))
    with pytest.raises(C.ValidationException, match="lacks \\['tmin'\\]"):
        ens.run_parameter_ensemble(st_u, {k: v for k, v in mem.items() if k != 'tmin'}, sets, output_vars=('q',))
    with pytest.raises(C.ValidationException, match='rows'):
        ens.run_parameter_ensemble(st_u, mem, sets[:, 1:], output_vars=('q',))
