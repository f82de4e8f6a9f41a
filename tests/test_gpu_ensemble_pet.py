"""The ensemble runner with Hargreaves-Samani, Thornthwaite and given PET, with and without routing: every member equals
the plug-in calls on that member alone (hargreaves_samani / thornthwaite.execute -> abcd_execute -> mrtm.route) bit for
bit, a tmin that is the member's hs_tmin crosses the link once, the output options work unchanged, and the
configurations that cannot run are refused."""

from types import SimpleNamespace

import numpy as np
import pytest

from util import bitwise_equal, max_rel

pytestmark = pytest.mark.gpu

SY, EY, M = 1991, 1993, 36          # 1992 is a leap year
RTOL = 1e-9
ALL_VARS = ('pet', 'aet', 'q', 'soilmoisture', 'chstorage', 'avgchflow')
UNROUTED_VARS = ALL_VARS[:4]


@pytest.fixture(scope='module')
def world():
    from xanthos_b200 import synthetic, ensemble as ens
    from xanthos_b200.routing import mrtm
    from oracle.calendar_utils import set_month_arrays
    w = synthetic.make_world(24, 48, 700, 6, seed=31)
    s = w.settings()
    um = mrtm.upstream_genmatrix(mrtm.upstream(w.coords, mrtm.downstream(w.coords, w.flow_dir, s), s))
    nd = set_month_arrays(M, SY, EY)[:, 2]
    members = {'hs': [], 'thornthwaite': [], 'none': []}
    pars = None
    for k in range(3):
        ab = synthetic.abcd_inputs(w, M, seed=20 + k, with_pet=True)      # precip keeps its NaN, as the loader does
        pars = ab['pars'] if pars is None else pars
        hs = synthetic.hs_inputs(w, SY, EY, seed=40 + k)                  # NaN kept in hs_*
        members['hs'].append(dict(hs, precip=ab['precip'], tmin=ab['tmin']))
        tw = synthetic.thornthwaite_inputs(w, SY, EY, seed=50 + k)
        members['thornthwaite'].append(dict(tair=tw['tair'], precip=ab['precip'], tmin=ab['tmin']))
        members['none'].append(dict(pet=ab['pet'], precip=ab['precip'], tmin=ab['tmin']))
    assert np.isnan(members['hs'][0]['hs_tas']).any() and np.isnan(members['hs'][0]['precip']).any()
    pm = synthetic.pm_inputs(w, SY, EY, nlcs=8, seed=10)
    pm_statics = dict(pm_tables={k: v for k, v in pm.items() if k not in ens.PM_FORCING + ('lct_load', 'tairprev_load')},
                      lct_load=pm['lct_load'], elev=pm['elev'], water_idx=pm['water_idx'], snow_idx=pm['snow_idx'],
                      lc_years=pm['lc_years'], nlcs=8)
    pm_member = {k: np.nan_to_num(pm[k]) for k in ens.PM_FORCING}
    pm_member['precip'], pm_member['tmin'] = members['none'][0]['precip'], members['none'][0]['tmin']
    return SimpleNamespace(w=w, um=um, nd=nd, pars=pars, members=members, pm_statics=pm_statics, pm_member=pm_member)


def statics_kw(wd, model, routing, **over):
    """Keyword arguments of EnsembleStatics for PET model `model`: PM arguments only for 'pm', routing arguments only
    with routing; `over` replaces any of them."""
    w = wd.w
    kw = dict(ncell=w.ncell, start_yr=SY, end_yr=EY, pm_tables=None, lct_load=None, elev=None, water_idx=None,
              snow_idx=None, lc_years=None, nlcs=None, n_basins=w.n_basins, basin_ids=w.basin_ids, abcd_pars=wd.pars,
              area=w.area, flow_dist=None, velocity=None, upstream_matrix=None, ndays=None, dt=10800, runoff_spinup=M,
              routing_spinup=6, pet=model, latitude=w.coords[:, 2] if model in ('hs', 'thornthwaite') else None,
              routing=routing)
    if routing:
        kw.update(flow_dist=w.flow_dist, velocity=w.velocity, upstream_matrix=wd.um, ndays=wd.nd)
    if model == 'pm':
        kw.update(wd.pm_statics)
    kw.update(over)
    return kw


def statics(wd, pet, routing):
    from xanthos_b200 import ensemble as ens
    return ens.EnsembleStatics(**statics_kw(wd, pet, routing))


def standalone(wd, mem, pet, routing):
    """The member through the plug-in calls, with the loader's nan_to_num on ABCD's tmin."""
    from xanthos_b200.pet import hargreaves_samani, thornthwaite
    from xanthos_b200.runoff import abcd
    from xanthos_b200.routing import mrtm
    w = wd.w
    if pet == 'hs':
        data = SimpleNamespace(coords=w.coords, hs_tas=mem['hs_tas'], hs_tmax=mem['hs_tmax'], hs_tmin=mem['hs_tmin'])
        p = hargreaves_samani.execute(SimpleNamespace(StartYear=SY), data)
    elif pet == 'thornthwaite':
        p = thornthwaite.execute(mem['tair'], np.radians(w.coords[:, 2]), SY, EY)
    else:
        p = mem['pet']
    pet_h, aet, q, sav = abcd.abcd_execute(w.n_basins, w.basin_ids, p, mem['precip'], np.nan_to_num(mem['tmin']),
                                           wd.pars, M, M, -1)
    out = {'pet': pet_h, 'aet': aet, 'q': q, 'soilmoisture': sav}
    if routing:
        chs, avg, _ = mrtm.route(wd.um, q, w.flow_dist, w.velocity, w.area, wd.nd, 10800, 6)
        out.update(chstorage=chs, avgchflow=avg)
    return out


def check_members(wd, res, members, pet, routing, output_vars):
    w = wd.w
    rows = 2 if routing else 1
    assert res['basin_aggregates'].shape == (len(members), rows, M, w.n_basins)
    want_cache = {}
    for k, mem in enumerate(members):
        if id(mem) not in want_cache:
            want_cache[id(mem)] = standalone(wd, mem, pet, routing)
        want = want_cache[id(mem)]
        for v in output_vars:
            assert bitwise_equal(res[k][v], want[v]), (k, v)
        for b in range(w.n_basins):
            idx = w.basin_ids == b + 1
            q_b = np.nansum(want['q'][idx] * (w.area[idx] * 1e-6)[:, None], axis=0)
            assert max_rel(res['basin_aggregates'][k, 0, :, b], q_b, floor=1e-12) < 1e-12
            if routing:
                f_b = np.nansum(want['avgchflow'][idx], axis=0)
                assert max_rel(res['basin_aggregates'][k, 1, :, b], f_b, floor=1e-12) < 1e-12
    return want_cache


def test_hs_routed_equals_the_plugin_calls(world):
    from xanthos_b200 import ensemble as ens
    from oracle import pet as opet
    members = world.members['hs']
    res = ens.run_ensemble(statics(world, 'hs', True), members, output_vars=('pet', 'q', 'avgchflow', 'chstorage'))
    check_members(world, res, members, 'hs', True, ('pet', 'q', 'avgchflow', 'chstorage'))
    m = members[1]
    want = opet.hs_pet(m['hs_tas'], m['hs_tmax'], m['hs_tmin'], world.w.coords[:, 2], SY, EY)
    assert max_rel(res[1]['pet'], want, floor=1e-6) < RTOL


def test_hs_unrouted_nine_members_and_routed_outputs_refused(world):
    from xanthos_b200 import ensemble as ens, _cuda as C
    st = statics(world, 'hs', False)
    members = [world.members['hs'][i % 3] for i in range(9)]      # odd count: the staging ring and pinned pool reused
    res = ens.run_ensemble(st, members, output_vars=UNROUTED_VARS)
    check_members(world, res, members, 'hs', False, UNROUTED_VARS)
    assert res['basin_aggregates'].shape == (9, 1, M, world.w.n_basins)
    assert ens.EnsembleRunner(st, ('q',)).group == 1
    uploaded = []

    def member(k):
        def load():
            uploaded.append(k)
            return members[k]
        return load
    for bad in (('q', 'avgchflow'), ('chstorage',)):
        with pytest.raises(C.ValidationException, match='routing'):
            ens.EnsembleRunner(st, bad)
        with pytest.raises(C.ValidationException, match='routing'):
            ens.run_ensemble(st, [member(k) for k in range(3)], output_vars=bad)
    assert uploaded == []


@pytest.mark.parametrize("routing", [True, False])
def test_thornthwaite_equals_the_plugin_calls(world, routing):
    from xanthos_b200 import ensemble as ens
    from oracle import pet as opet
    members = world.members['thornthwaite']
    out_vars = ALL_VARS if routing else UNROUTED_VARS
    res = ens.run_ensemble(statics(world, 'thornthwaite', routing), members, output_vars=out_vars)
    check_members(world, res, members, 'thornthwaite', routing, out_vars)
    want = opet.thornthwaite_pet(members[2]['tair'], np.radians(world.w.coords[:, 2]), SY, EY)
    assert max_rel(res[2]['pet'], want, floor=1e-6) < RTOL


@pytest.mark.parametrize("routing", [True, False])
def test_given_pet_equals_abcd_of_that_pet(world, routing):
    from xanthos_b200 import ensemble as ens
    members = world.members['none']
    out_vars = ALL_VARS if routing else UNROUTED_VARS
    res = ens.run_ensemble(statics(world, 'none', routing), members, output_vars=out_vars)
    check_members(world, res, members, 'none', routing, out_vars)
    for k, mem in enumerate(members):
        assert bitwise_equal(res[k]['pet'], mem['pet'])


def test_tmin_shared_with_hs_tmin_crosses_the_link_once(world):
    from xanthos_b200 import ensemble as ens
    w, st = world.w, statics(world, 'hs', False)
    rng = np.random.default_rng(7)
    members = []
    for m in world.members['hs']:
        mem = {k: m[k].copy() for k in ('hs_tas', 'hs_tmax', 'hs_tmin', 'precip')}
        mem['hs_tmin'].ravel()[rng.choice(mem['hs_tmin'].size, 40, replace=False)] = np.nan
        mem['tmin'] = mem['hs_tmin']                                       # one array: TempMinFile is hs_tmin
        members.append(mem)
    field = 8 * w.ncell * M
    res = ens.run_ensemble(st, members, output_vars=UNROUTED_VARS)
    check_members(world, res, members, 'hs', False, UNROUTED_VARS)     # ABCD read tmin as np.nan_to_num(hs_tmin)
    assert res['stats']['h2d_bytes'] == 4 * field * len(members)
    apart = [dict(m, tmin=m['tmin'].copy()) for m in members]           # the same values in two arrays: five fields
    res_apart = ens.run_ensemble(st, apart, output_vars=UNROUTED_VARS)
    assert res_apart['stats']['h2d_bytes'] == 5 * field * len(members)
    for k in range(len(members)):
        assert all(bitwise_equal(res_apart[k][v], res[k][v]) for v in UNROUTED_VARS)
    # single-precision values: the float32 copies keep the sharing and give the float64 run's results bit for bit
    m64 = []
    for mem in members:
        one = {k: mem[k].astype(np.float32).astype(np.float64) for k in ('hs_tas', 'hs_tmax', 'hs_tmin', 'precip')}
        one['tmin'] = one['hs_tmin']
        m64.append(one)
    packed = [ens.lossless_float32(m) for m in m64]
    assert all(p['tmin'] is p['hs_tmin'] and p['tmin'].dtype == np.float32 for p in packed)
    r64 = ens.run_ensemble(st, m64, output_vars=UNROUTED_VARS)
    r32 = ens.run_ensemble(st, packed, output_vars=UNROUTED_VARS)
    for k in range(len(members)):
        for v in UNROUTED_VARS:
            assert bitwise_equal(r32[k][v], r64[k][v]), (k, v)
    assert bitwise_equal(r32['basin_aggregates'], r64['basin_aggregates'])
    assert r64['stats']['h2d_bytes'] == 4 * field * len(members)
    assert r32['stats']['h2d_bytes'] == 4 * (field // 2) * len(members)
    assert r32['stats']['h2d_bytes'] < 0.6 * r64['stats']['h2d_bytes']


def test_output_options_without_routing(world):
    """Yearly km3 grids, basin sums, statistics, quantiles and drought of soil moisture on HS -> ABCD: what OutWriter,
    numpy and DroughtStats make of the stand-alone members' outputs, to the tolerances of the PM runner's tests."""
    from xanthos_b200 import ensemble as ens, _cuda as C
    from xanthos_b200.data_writer import out_writer
    from xanthos_b200.diagnostics.time_series import group_sum_device
    from xanthos_b200.drought.drought_stats import DroughtStats
    from oracle import ensemble_stats as es
    w, members = world.w, world.members['hs']
    out_vars, levels, years, nper = ('q', 'soilmoisture'), (0.05, 0.5, 0.95), (1992, 1993), 4
    spec = ens.OutputSpec(output_in_year=True, output_unit='km3', group_sums=('basin',), stats=ens.STATS,
                          quantiles=levels, drought=ens.DroughtSpec('soilmoisture', threshold_years=years, nper=nper))
    res = ens.run_ensemble(statics(world, 'hs', False), members, output_vars=out_vars, spec=spec)
    n, ny = len(members), M // 12
    assert res['basin_aggregates'].shape == (n, 1, M, w.n_basins)
    settings = SimpleNamespace(StartYear=SY, threshold_start_year=years[0], threshold_end_year=years[1],
                               threshold_nper=nper)
    stacks, dry = {v: [] for v in out_vars}, 0
    for k, mem in enumerate(members):
        monthly = standalone(world, mem, 'hs', False)
        for v in out_vars:
            a = out_writer.agg_to_year(C.remember(np.array(monthly[v]), C.Field.from_host(monthly[v])), 'sum')
            a = np.asarray(a) * (np.asarray(w.area) / 1e6)[:, None]
            assert res[k][v].shape == (w.ncell, ny) and bitwise_equal(res[k][v], a), (k, v)
            stacks[v].append(a)
            if v == 'q':
                basin = group_sum_device(w.basin_ids, C.Field.from_host(a).t).cpu().numpy()
                assert bitwise_equal(res[k]['group_sums']['basin'], basin)
                assert bitwise_equal(res['group_sums']['basin'][k], basin)
        x = np.ascontiguousarray(monthly['soilmoisture'].T)
        th = DroughtStats.calculate_thresholds(x, settings)
        S_, I_, D_ = DroughtStats.droughtstats(None, x, th)
        got = res[k]['drought']
        assert bitwise_equal(got['thresholds'], th)
        with np.errstate(invalid='ignore'):
            summ = np.stack([(D_ > 0).sum(0), (D_ == 1).sum(0), D_.max(0), S_.max(0)]).astype(np.float64)
        for i, name in enumerate(ens.DROUGHT_SUMMARY):
            assert bitwise_equal(got['summary'][name], summ[i]), (k, name)
        assert bitwise_equal(res['drought_summary'][k], summ)
        dry = dry + (D_ > 0).astype(np.int32)
    assert np.array_equal(res['ensemble_drought']['members_in_drought'], dry.T)
    assert bitwise_equal(res['ensemble_drought']['frequency'], dry.T / n)
    assert res['ensemble_stats']['n_members'] == n and res['ensemble_quantiles']['n_members'] == n
    for v in out_vars:
        x = np.stack(stacks[v])
        want = es.run(list(x), ddof=0)
        with np.errstate(invalid='ignore'):
            ref = {'mean': np.mean(x, axis=0), 'min': np.min(x, axis=0), 'max': np.max(x, axis=0)}
            std = np.std(x, axis=0)
        for st in ens.STATS:
            assert bitwise_equal(res['ensemble_stats'][v][st], want[st]), (v, st)
            if st in ref:
                assert bitwise_equal(res['ensemble_stats'][v][st], ref[st]), (v, st)
        ok = ~np.isnan(std)
        np.testing.assert_allclose(res['ensemble_stats'][v]['std'][ok], std[ok], rtol=1e-12,
                                   atol=1e-15 * np.nanmax(np.abs(x)))
        assert bitwise_equal(res['ensemble_quantiles'][v], np.quantile(x, levels, axis=0)), v


@pytest.mark.parametrize("pet,routing,over,names", [
    ('hargreaves', False, {}, 'unknown PET model'),
    ('hs', False, {'latitude': None}, 'latitude'),
    ('thornthwaite', True, {'latitude': None}, 'latitude'),
    ('hs', False, {'latitude': np.zeros(5)}, 'latitude has 5 entries'),
    ('pm', True, {'pm_tables': None}, 'pm_tables'),
    ('pm', True, {'lct_load': None, 'nlcs': None}, 'lct_load, nlcs'),
    ('pm', False, {'elev': None, 'lc_years': None}, 'elev, lc_years'),
    ('hs', True, {'upstream_matrix': None}, 'upstream_matrix'),
    ('none', True, {'flow_dist': None, 'ndays': None}, 'flow_dist, ndays'),
    ('thornthwaite', True, {'velocity': None, 'latitude': None}, 'velocity, latitude'),
])
def test_statics_refuse_what_cannot_run(world, pet, routing, over, names):
    from xanthos_b200 import ensemble as ens, _cuda as C
    with pytest.raises(C.ValidationException, match=names):
        # every other argument of a runnable `pet` configuration given: only the pieces in `over` are missing
        ens.EnsembleStatics(**statics_kw(world, pet if pet in ens.PET_MODELS else 'hs', routing, pet=pet, **over))


def test_pm_statics_with_the_new_keywords_at_their_defaults(world):
    """The PM positional call and the same call with pet='pm', latitude=None, routing=True give the plug-in results
    bitwise and upload the same eight fields."""
    from xanthos_b200 import ensemble as ens
    from xanthos_b200.pet import penman_monteith as pm_mod
    from xanthos_b200.runoff import abcd
    from xanthos_b200.routing import mrtm
    w, ps, mem = world.w, world.pm_statics, world.pm_member
    args = (w.ncell, SY, EY, ps['pm_tables'], ps['lct_load'], ps['elev'], ps['water_idx'], ps['snow_idx'],
            ps['lc_years'], 8, w.n_basins, w.basin_ids, world.pars, w.area, w.flow_dist, w.velocity, world.um,
            world.nd, 10800, M, 6)
    plain = ens.run_ensemble(ens.EnsembleStatics(*args), [mem], output_vars=ALL_VARS)
    keyed = ens.run_ensemble(ens.EnsembleStatics(*args, pet='pm', latitude=None, routing=True), [mem],
                             output_vars=ALL_VARS)
    data = SimpleNamespace(**{**ps['pm_tables'], 'lct_load': ps['lct_load'], 'elev': ps['elev'], **mem})
    pet = pm_mod.run_pmpet(data, w.ncell, 8, SY, EY, ps['water_idx'], ps['snow_idx'], ps['lc_years'])
    _, aet, q, sav = abcd.abcd_execute(w.n_basins, w.basin_ids, pet, mem['precip'], mem['tmin'], world.pars, M, M, -1)
    chs, avg, _ = mrtm.route(world.um, q, w.flow_dist, w.velocity, w.area, world.nd, 10800, 6)
    want = {'pet': pet, 'aet': aet, 'q': q, 'soilmoisture': sav, 'chstorage': chs, 'avgchflow': avg}
    for res in (plain, keyed):
        for v in ALL_VARS:
            assert bitwise_equal(res[0][v], want[v]), v
        assert res['basin_aggregates'].shape == (1, 2, M, w.n_basins)
        assert res['stats']['h2d_bytes'] == 8 * 8 * w.ncell * M
    assert bitwise_equal(plain['basin_aggregates'], keyed['basin_aggregates'])
