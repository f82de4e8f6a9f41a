"""The ensemble runner's output options (OutputSpec): yearly / km3 grids and group sums reduced on the device, equal bit
for bit to what OutWriter produces from each member's monthly outputs, and the across-member statistics against numpy
and the numpy restatement of the kernels (oracle/ensemble_stats.py)."""

from types import SimpleNamespace

import numpy as np
import pytest

from util import bitwise_equal

pytestmark = pytest.mark.gpu

SY, EY, M = 1991, 1993, 36
VARS = ('q', 'avgchflow')


@pytest.fixture(scope='module')
def world():
    from xanthos_b200 import synthetic, ensemble as ens
    from xanthos_b200.routing import mrtm
    from oracle.calendar_utils import set_month_arrays
    w = synthetic.make_world(24, 48, 700, 6, seed=31)
    s = w.settings()
    um = mrtm.upstream_genmatrix(mrtm.upstream(w.coords, mrtm.downstream(w.coords, w.flow_dir, s), s))
    nd = set_month_arrays(M, SY, EY)[:, 2]
    rng = np.random.default_rng(5)
    members, pm0, ab0 = [], None, None
    for k in range(5):
        pm = synthetic.pm_inputs(w, SY, EY, nlcs=8, seed=10 + k)
        ab = synthetic.abcd_inputs(w, M, seed=20 + k, with_pet=False)
        mem = {key: np.nan_to_num(pm[key]) for key in ens.PM_FORCING}
        precip = ab['precip'].copy()
        if k in (1, 3):         # missing precipitation in some cells of two members: NaN in q from there on
            cells = rng.choice(w.ncell, 6, replace=False)
            precip[cells, rng.integers(0, M, 6)] = np.nan
        mem['precip'], mem['tmin'] = precip, np.nan_to_num(ab['tmin'])
        members.append(mem)
        if k == 0:
            pm0, ab0 = pm, ab
    country = (w.basin_ids % 4).astype(int)          # 0 = no country: left out of the sums
    country[rng.random(w.ncell) < 0.02] = 0
    region = (w.basin_ids % 2).astype(int) + 1
    tables = {k: v for k, v in pm0.items() if k not in ens.PM_FORCING + ('lct_load', 'tairprev_load')}
    args = (w.ncell, SY, EY, tables, pm0['lct_load'], pm0['elev'], pm0['water_idx'], pm0['snow_idx'], pm0['lc_years'],
            8, w.n_basins, w.basin_ids, ab0['pars'], w.area, w.flow_dist, w.velocity, um, nd, 10800, M, 6)
    st = ens.EnsembleStatics(*args, country_ids=country, region_ids=region)
    monthly = ens.run_ensemble(st, members, output_vars=VARS)
    assert any(np.isnan(monthly[k]['q']).any() for k in range(5)), "NaN precipitation must reach q"
    ids = {'basin': w.basin_ids, 'country': country, 'region': region}
    return SimpleNamespace(w=w, st=st, args=args, members=members, monthly=monthly, ids=ids)


def expected(wd, k, spec):
    """What OutWriter.write / write_aggregates make of member k's monthly outputs (as resident arrays, the device
    path): {var: [ncell, ntime]}, {scale: [ngroups, ntime]}."""
    from xanthos_b200 import _cuda as C
    from xanthos_b200.data_writer import out_writer
    from xanthos_b200.diagnostics.time_series import group_sum_device
    out = {}
    for v in VARS:
        a = wd.monthly[k][v]
        if spec.output_in_year:
            a = out_writer.agg_to_year(C.remember(np.array(a), C.Field.from_host(a)), 'mean' if v == 'avgchflow' else 'sum')
        if spec.output_unit == 'km3' and v != 'avgchflow':
            a = a * (np.asarray(wd.w.area) / 1e6)[:, None]
        out[v] = np.asarray(a)
    groups = {g: group_sum_device(wd.ids[g], C.Field.from_host(out['q']).t).cpu().numpy() for g in spec.group_sums}
    return out, groups


def check_stats(got, stacks, spec):
    from oracle import ensemble_stats as es
    for v in VARS:
        x = stacks[v]
        want = es.run(list(x), ddof=spec.ddof)
        with np.errstate(invalid='ignore'):
            ref = {'mean': np.mean(x, axis=0), 'min': np.min(x, axis=0), 'max': np.max(x, axis=0),
                   'std': np.std(x, axis=0, ddof=spec.ddof)}
        assert set(got[v]) == set(spec.stats)
        for st in spec.stats:
            assert bitwise_equal(got[v][st], want[st]), (v, st)
            if st == 'std':
                assert np.array_equal(np.isnan(got[v][st]), np.isnan(ref[st]))
                ok = ~np.isnan(ref[st])
                # atol: where the members agree to the last bits both formulas give rounding noise around 0
                np.testing.assert_allclose(got[v][st][ok], ref[st][ok], rtol=1e-12,
                                           atol=1e-15 * np.nanmax(np.abs(x)))
            else:
                assert bitwise_equal(got[v][st], ref[st]), (v, st)
        assert np.isnan(x).any() == np.isnan(got[v]['mean']).any()


@pytest.mark.parametrize("yearly,ddof", [(True, 0), (False, 1)])
def test_reduced_members_and_stats_equal_out_writer_and_numpy(world, yearly, ddof):
    """Yearly + km3 and monthly + km3 with basin / country / region sums and all four statistics: every member's grids
    and group sums are bitwise OutWriter's; mean / min / max bitwise numpy over the stacked members, every statistic
    bitwise the oracle, std within 1e-12 of numpy.std; avgchflow is the yearly mean and never converted."""
    from xanthos_b200 import ensemble as ens
    spec = ens.OutputSpec(output_in_year=yearly, output_unit='km3', group_sums=('basin', 'country', 'region'),
                          stats=ens.STATS, ddof=ddof)
    res = ens.run_ensemble(world.st, world.members, output_vars=VARS, spec=spec)
    ntime = M // 12 if yearly else M
    stacks = {v: [] for v in VARS}
    for k in range(5):
        fields, groups = expected(world, k, spec)
        for v in VARS:
            assert res[k][v].shape == (world.w.ncell, ntime)
            assert bitwise_equal(res[k][v], fields[v]), (k, v)
            stacks[v].append(fields[v])
        for g in spec.group_sums:
            assert bitwise_equal(res[k]['group_sums'][g], groups[g]), (k, g)
            assert bitwise_equal(res['group_sums'][g][k], groups[g]), (k, g)
            assert res['group_sums'][g].shape == (5, int(world.ids[g].max()), ntime)
    # the monthly avgchflow comes back untouched, the monthly basin aggregates are still there
    if not yearly:
        for k in range(5):
            assert bitwise_equal(res[k]['avgchflow'], world.monthly[k]['avgchflow'])
    assert bitwise_equal(res['basin_aggregates'], world.monthly['basin_aggregates'])
    assert res['ensemble_stats']['n_members'] == 5
    check_stats(res['ensemble_stats'], {v: np.stack(stacks[v]) for v in VARS}, spec)


def test_member_fields_off_copies_back_group_sums_and_stats_only(world):
    from xanthos_b200 import ensemble as ens
    kw = dict(output_in_year=True, output_unit='km3', group_sums=('basin', 'region'), stats=('mean', 'max'))
    res = ens.run_ensemble(world.st, world.members, output_vars=VARS, aggregates=False,
                           spec=ens.OutputSpec(member_fields=False, **kw))
    full = ens.run_ensemble(world.st, world.members, output_vars=VARS, aggregates=False, spec=ens.OutputSpec(**kw))
    ny, nc = M // 12, world.w.ncell
    for k in range(5):
        assert set(res[k]) == {'group_sums'}
        for g in kw['group_sums']:
            assert bitwise_equal(res[k]['group_sums'][g], full[k]['group_sums'][g])
    for v in VARS:
        for st in kw['stats']:
            assert bitwise_equal(res['ensemble_stats'][v][st], full['ensemble_stats'][v][st])
    groups = sum(int(world.ids[g].max()) for g in kw['group_sums'])
    want = 8 * (5 * groups * ny + len(VARS) * len(kw['stats']) * nc * ny)
    assert res['stats']['d2h_bytes'] == want
    assert full['stats']['d2h_bytes'] == want + 8 * 5 * len(VARS) * nc * ny


def test_partial_stats_merged_on_the_device_equal_the_oracle_merge(world):
    """Members {0, 1, 2} and {3, 4} accumulated by two runners and merged with xan_ens_stats_merge: bitwise the
    oracle's merge of the same partials; min / max bitwise the single run."""
    from xanthos_b200 import ensemble as ens
    from oracle import ensemble_stats as es
    spec = ens.OutputSpec(output_in_year=True, stats=ens.STATS, ddof=1)
    whole = ens.run_ensemble(world.st, world.members, output_vars=VARS, aggregates=False, spec=spec)['ensemble_stats']
    ra = ens.EnsembleRunner(world.st, VARS, aggregates=False, spec=spec)
    rb = ens.EnsembleRunner(world.st, VARS, aggregates=False, spec=spec)
    list(ra.run(world.members[:3]))
    list(rb.run(world.members[3:]))
    got = ra.finalize_stats(ra.merge_stats(ra.stats_partial(), 3, rb.stats_partial(), 2), 5)
    for v in VARS:
        x = [expected(world, k, spec)[0][v] for k in range(5)]
        pa, pb = None, None
        for j in range(3):
            pa = es.update(pa, x[j], j + 1)
        for j in range(2):
            pb = es.update(pb, x[3 + j], j + 1)
        want = es.finalize(es.merge(pa, 3, pb, 2), 5, ddof=1)
        for st in ens.STATS:
            assert bitwise_equal(got[v][st], want[st]), (v, st)
        assert bitwise_equal(got[v]['min'], whole[v]['min']) and bitwise_equal(got[v]['max'], whole[v]['max'])


def test_spec_validation_on_the_runner(world):
    from xanthos_b200 import ensemble as ens, _cuda as C
    with pytest.raises(C.ValidationException):
        ens.EnsembleRunner(world.st, ('q', 'chstorage'), spec=ens.OutputSpec(output_in_year=True))
    with pytest.raises(C.ValidationException):
        ens.EnsembleRunner(world.st, ('chstorage',), spec=ens.OutputSpec(output_unit='km3'))
    ens.EnsembleRunner(world.st, ('chstorage',), spec=ens.OutputSpec(stats=('mean',)))      # monthly mm: allowed
    bare = ens.EnsembleStatics(*world.args)
    with pytest.raises(C.ValidationException):
        ens.EnsembleRunner(bare, VARS, spec=ens.OutputSpec(group_sums=('country',)))
    short = ens.EnsembleStatics(*world.args, region_ids=world.ids['region'][:-1])
    with pytest.raises(C.ValidationException):
        ens.EnsembleRunner(short, VARS, spec=ens.OutputSpec(group_sums=('region',)))
