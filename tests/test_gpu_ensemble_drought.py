"""Drought statistics in the ensemble runner: xan_drought_scan against oracle.postproc.droughtstats and
xan_drought_stats bit for bit, and OutputSpec(drought=DroughtSpec(...)) against DroughtStats on every member's
plug-in outputs and numpy over the members."""

from types import SimpleNamespace

import numpy as np
import pytest

from util import bitwise_equal
from test_gpu_ensemble_quantiles import world, SY, EY, M  # noqa: F401  (the synthetic world with missing precipitation)

pytestmark = pytest.mark.gpu

NCELL, NMONTHS = 203, 37          # 37 months: not a multiple of the kernel's load batch


def _case(n, nthresh, seed):
    """n members' fields [n, NMONTHS, NCELL] and thresholds [nthresh, NCELL] with NaN in both, a drought from month 0
    (cell 0), one running through the last month (cell 1), a +inf threshold (cell 2: NaN severity) and a threshold
    below every value (cell 3: never dry)."""
    rng = np.random.default_rng(seed)
    th = rng.uniform(2.0, 6.0, (nthresh, NCELL))
    th[rng.random(th.shape) < 0.02] = np.nan
    th[:, 2], th[:, 3] = np.inf, -1.0
    h = rng.uniform(0.0, 10.0, (n, NMONTHS, NCELL))
    h[rng.random(h.shape) < 0.03] = np.nan
    h[:, :5, 0] = 0.5
    h[:, NMONTHS - 6:, 1] = 0.25
    h[:, :, 4] = np.nan
    th[:, :2] = 3.0
    return h, th


def _poisoned(x, ld, fill=np.nan, dtype=None):
    """host [rows, NCELL] -> cuda [rows, ld] with the padding columns set to `fill`."""
    import torch
    t = torch.full((x.shape[0], ld), fill, dtype=dtype or torch.float64, device='cuda')
    t[:, :NCELL] = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return t


@pytest.mark.parametrize("nthresh", [1, 4, 12])
@pytest.mark.parametrize("n", [1, 5, 64])
def test_scan_equals_oracle_and_drought_stats_bitwise(n, nthresh):
    import torch
    from oracle import postproc as ref
    from xanthos_b200 import _cuda as C
    from xanthos_b200.drought.drought_stats import drought_scan_device, droughtstats_device
    h, th = _case(n, nthresh, seed=100 * n + nthresh)
    ld = C.padded_ld(NCELL)
    d_th = _poisoned(th, ld)
    count = torch.full((NMONTHS, ld), -7, dtype=torch.int32, device='cuda')     # padding must stay -7
    count[:, :NCELL] = 0
    count_only = count.clone()
    want_count = np.zeros((NMONTHS, NCELL), dtype=np.int64)
    for k in range(n):
        S_, I_, D_ = ref.droughtstats(h[k], th)
        d_h = _poisoned(h[k], ld)
        sid = [torch.full((NMONTHS, ld), -3.0, dtype=torch.float64, device='cuda') for _ in range(3)]
        summary = torch.full((4, ld), -5.0, dtype=torch.float64, device='cuda')
        summary_only = summary.clone()
        drought_scan_device(d_h, NCELL, d_th, sid, count, summary)
        drought_scan_device(d_h, NCELL, d_th, None, count_only, summary_only)
        stats = droughtstats_device(d_h, NCELL, d_th)
        for got, old, want in zip(sid, stats, (S_, I_, D_)):
            assert bitwise_equal(got[:, :NCELL].cpu().numpy(), want)
            assert bitwise_equal(got[:, :NCELL].cpu().numpy(), old[:, :NCELL].cpu().numpy())
        with np.errstate(invalid='ignore'):
            want_summary = np.stack([(D_ > 0).sum(0), (D_ == 1).sum(0), D_.max(0), S_.max(0)]).astype(np.float64)
        for s in (summary, summary_only):
            assert bitwise_equal(s[:, :NCELL].cpu().numpy(), want_summary), k
            assert (s[:, NCELL:] == -5.0).all()
        want_count += D_ > 0
    assert np.isnan(want_summary[3, 2]) and want_summary[3, 3] == 0.0 and want_summary[0, 3] == 0.0
    assert want_summary[0, 0] >= 5 and D_[0, 0] == 1.0 and D_[-1, 1] >= 6.0          # edges present in the case
    for c in (count, count_only):
        got = c.cpu().numpy()
        assert np.array_equal(got[:, :NCELL], want_count) and (got[:, NCELL:] == -7).all()


def test_scan_refuses_bad_calls():
    import torch
    from xanthos_b200 import _cuda as C
    x = torch.zeros((4, 16), dtype=torch.float64, device='cuda')
    cnt = torch.zeros((4, 16), dtype=torch.int32, device='cuda')
    lib, p, st = C.lib(), C.ptr, C.stream_ptr()
    assert lib.xan_drought_scan(p(x), p(x), 10, 4, 16, 1, 16, None, None, None, None, None, st) == C.XAN_E_INVALID
    assert lib.xan_drought_scan(p(x), p(x), 10, 4, 16, 1, 16, p(x), None, None, None, None, st) == C.XAN_E_INVALID
    assert lib.xan_drought_scan(p(x), p(x), 10, 4, 16, 1, 16, None, None, None, p(cnt), None, st) == C.XAN_E_INVALID
    assert lib.xan_drought_scan(p(x), p(x), 10, 4, 16, 1, 16, None, None, None, p(cnt), p(x), st) == C.XAN_OK
    torch.cuda.synchronize()


# ---- the runner ----------------------------------------------------------------------------------------------------
VARS = ('q', 'avgchflow')
YEARS, NPER = (1992, 1993), 4      # the reference's slice [12:24]: one year, three samples per period of 3 months


@pytest.fixture(scope='module')
def plugin(world):  # noqa: F811
    """Every member's monthly q and soil moisture as the plug-in path returns them, [ncell, nmonths]."""
    from xanthos_b200 import ensemble as ens
    monthly = ens.run_ensemble(world.st, world.members, output_vars=('q', 'soilmoisture'), aggregates=False)
    return {v: [monthly[k][v] for k in range(5)] for v in ('q', 'soilmoisture')}


def _shared_thresholds(world, plugin, var):  # noqa: F811
    """Thresholds of member 0 with a +inf and a NaN cell (NaN severity, never dry)."""
    from oracle import postproc as ref
    th = ref.getthresh(plugin[var][0].T[:24], 12)
    th[:, 5], th[3, 9] = np.inf, np.nan
    return th


def _reference(world, plugin, var, th):  # noqa: F811
    """(thresholds, S, I, D) of every member through DroughtStats, [nmonths, ncell] each."""
    from xanthos_b200.drought.drought_stats import DroughtStats
    settings = SimpleNamespace(StartYear=SY, threshold_start_year=YEARS[0], threshold_end_year=YEARS[1],
                               threshold_nper=NPER)
    out = []
    for k in range(5):
        x = np.ascontiguousarray(plugin[var][k].T)
        t = DroughtStats.calculate_thresholds(x, settings) if th is None else th
        out.append((t,) + DroughtStats.droughtstats(None, x, t))
    return out


@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("var", ['q', 'soilmoisture'])
def test_runner_drought_equals_drought_stats_per_member(world, plugin, var, shared):  # noqa: F811
    from oracle import postproc as ref
    from xanthos_b200 import ensemble as ens
    th = _shared_thresholds(world, plugin, var) if shared else None
    d = ens.DroughtSpec(var, thresholds=th, threshold_years=None if shared else YEARS, nper=NPER, fields=True)
    res = ens.run_ensemble(world.st, world.members, output_vars=VARS, aggregates=False,
                           spec=ens.OutputSpec(member_fields=False, drought=d))
    want = _reference(world, plugin, var, th)
    ncell = world.w.ncell
    for k, (t, S_, I_, D_) in enumerate(want):
        got = res[k]['drought']
        assert set(got) == {'summary', 'severity', 'intensity', 'duration'} | (set() if shared else {'thresholds'})
        assert 'q' not in res[k]
        if not shared:
            assert got['thresholds'].shape == (NPER, ncell)
            assert bitwise_equal(got['thresholds'], t)
            assert bitwise_equal(t, ref.calculate_thresholds(plugin[var][k].T, SY, YEARS[0], YEARS[1], NPER))
        for name, x in zip(ens.DROUGHT_FIELDS, (S_, I_, D_)):
            assert got[name].shape == (ncell, M) and bitwise_equal(got[name], x.T), (k, name)
        with np.errstate(invalid='ignore'):
            summ = np.stack([(D_ > 0).sum(0), (D_ == 1).sum(0), D_.max(0), S_.max(0)]).astype(np.float64)
        for i, name in enumerate(ens.DROUGHT_SUMMARY):
            assert bitwise_equal(got['summary'][name], summ[i]), (k, name)
        assert bitwise_equal(res['drought_summary'][k], summ)                # member order
    counts = sum((D_ > 0).astype(np.int32) for _, _, _, D_ in want).T
    ed = res['ensemble_drought']
    assert ed['n_members'] == 5 and ed['members_in_drought'].dtype == np.int32
    assert np.array_equal(ed['members_in_drought'], counts)
    assert bitwise_equal(ed['frequency'], counts / 5)
    assert res['drought_summary'].shape == (5, 4, ncell)
    assert counts.max() > 0 and (counts < 5).any()
    if shared:
        assert np.isnan(res['drought_summary'][:, 3, 5]).all() and (counts[9, 3::12] == 0).all()


def test_drought_leaves_every_other_output_unchanged_and_adds_its_bytes(world):  # noqa: F811
    from xanthos_b200 import ensemble as ens
    kw = dict(output_in_year=True, output_unit='km3', group_sums=('basin',), stats=('mean', 'std', 'min', 'max'),
              quantiles=(0.1, 0.5, 0.9))
    base = ens.run_ensemble(world.st, world.members, output_vars=VARS, spec=ens.OutputSpec(**kw))
    d = ens.DroughtSpec('q', threshold_years=YEARS, nper=NPER, fields=True)
    res = ens.run_ensemble(world.st, world.members, output_vars=VARS, spec=ens.OutputSpec(drought=d, **kw))
    assert set(res) == set(base) | {'drought_summary', 'ensemble_drought'}
    for k in range(5):
        assert set(res[k]) == set(base[k]) | {'drought'}
        for key in base[k]:
            if key == 'group_sums':
                assert all(bitwise_equal(res[k][key][g], base[k][key][g]) for g in base[k][key])
            else:
                assert bitwise_equal(res[k][key], base[k][key]), (k, key)
    assert bitwise_equal(res['basin_aggregates'], base['basin_aggregates'])
    assert bitwise_equal(res['group_sums']['basin'], base['group_sums']['basin'])
    for v in VARS:
        for st in kw['stats']:
            assert bitwise_equal(res['ensemble_stats'][v][st], base['ensemble_stats'][v][st]), (v, st)
        assert bitwise_equal(res['ensemble_quantiles'][v], base['ensemble_quantiles'][v]), v
    from xanthos_b200 import _cuda as C
    ncell, ld = world.w.ncell, C.padded_ld(world.w.ncell)
    per_member = 8 * 4 * ld + 8 * NPER * ncell + 3 * 8 * ncell * M      # summary, thresholds, S / I / D
    assert res['stats']['d2h_bytes'] == base['stats']['d2h_bytes'] + 5 * per_member + 4 * ncell * M


def test_two_runners_combine(world):  # noqa: F811
    from xanthos_b200 import ensemble as ens
    spec = ens.OutputSpec(member_fields=False, drought=ens.DroughtSpec('soilmoisture', threshold_years=YEARS, nper=NPER))
    whole = ens.run_ensemble(world.st, world.members, output_vars=VARS, aggregates=False, spec=spec)
    ra = ens.EnsembleRunner(world.st, VARS, aggregates=False, spec=spec)
    rb = ens.EnsembleRunner(world.st, VARS, aggregates=False, spec=spec)
    sa = [r['drought']['summary'] for _, r in ra.run(world.members[:3])]
    sb = [r['drought']['summary'] for _, r in rb.run(world.members[3:])]
    for k, s in enumerate(sa + sb):
        assert bitwise_equal(np.stack([s[n] for n in ens.DROUGHT_SUMMARY]), whole['drought_summary'][k])
    part = ens.merge_drought_counts(ra.drought_partial(), 3, rb.drought_partial(), 2)
    got = ra.finalize_drought(part, 5)
    assert got['n_members'] == 5
    assert np.array_equal(got['members_in_drought'], whole['ensemble_drought']['members_in_drought'])
    assert bitwise_equal(got['frequency'], whole['ensemble_drought']['frequency'])


def test_invalid_drought_specs_refused_before_any_upload(world):  # noqa: F811
    from xanthos_b200 import ensemble as ens, _cuda as C
    uploaded = []

    def member(k):
        def load():
            uploaded.append(k)
            return world.members[k]
        return load
    bad = [ens.DroughtSpec('q', thresholds=np.ones((12, world.w.ncell - 1))),       # wrong cell count
           ens.DroughtSpec('q', threshold_years=(SY - 1, EY)),                     # outside the run
           ens.DroughtSpec('q', threshold_years=(EY, EY)),                         # slice [24:12] is empty
           ens.DroughtSpec('q', threshold_years=YEARS, nper=5)]                    # 12 months, 5 periods
    for d in bad:
        with pytest.raises(C.ValidationException):
            ens.run_ensemble(world.st, [member(k) for k in range(5)], output_vars=VARS, aggregates=False,
                             spec=ens.OutputSpec(drought=d))
    assert uploaded == []
