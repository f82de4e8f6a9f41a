"""
GPU tests of the PET, runoff, layout and aggregation kernels at the edges of their shapes and values, called through
the C entry points and compared with the numpy oracle.

Every call goes through `guarded`: it runs at three row pitches (ld = ncell, padded_ld(ncell), padded_ld(ncell) + 16),
allocates every array with one extra row, fills the padding columns and the extra row of inputs with NaN and those of
outputs with a signalling-NaN bit pattern no kernel computes, and checks that the output padding still holds that
pattern and that the results equal, bit for bit, those of the same call with zero padding (and those at the other
pitches).  A kernel that reads padding or writes past its rows fails an assertion; every access stays inside the
allocation, so no indexing error can fault.

Tolerances are the ones the kernels' headers claim: 1e-9 relative with a 1e-6 floor and an exact zero / NaN pattern
for Hargreaves-Samani, Thornthwaite, Hargreaves and GWAM; 1e-12 for the exact-order Penman-Monteith kernel and 1e-11
for the fast one; bit for bit where the kernel keeps numpy's operation order (layout, group and year sums, drought
thresholds, ABCD with zero PET and one cell per basin); 1e-9 for ABCD basins of several cells (block reduction of the
re-initialisation), 1e-12 for the warp-tree basin sums and 1e-13 for the yearly aggregation (pandas adds with
compensation).
"""

import ctypes
import math

import numpy as np
import pytest

from util import max_rel

pytestmark = pytest.mark.gpu

RTOL = 1e-9
NAN_BITS = 0x7FF8000000000000           # quiet NaN: padding of inputs
F32_NAN_BITS = 0x7FC00000
GUARD_BITS = 0x7FF4DEADBEEF0BAD         # signalling NaN: padding of outputs; arithmetic never produces it


# ---- guarded-buffer harness -------------------------------------------------------------------------------------------

class In:
    """Input of a guarded call: `a` [rows, cols]; pitched arrays are stored with row pitch ld, others with cols."""

    def __init__(self, a, pitched=True):
        self.a = np.ascontiguousarray(a)
        assert self.a.ndim == 2 and self.a.dtype in (np.float64, np.float32)
        self.rows, self.cols = self.a.shape
        self.pitched = pitched


class Out:
    """Output of a guarded call: [rows, cols] float64; `init` [rows, cols] for an array updated in place."""

    def __init__(self, rows, cols, pitched=True, init=None):
        self.rows, self.cols, self.pitched = int(rows), int(cols), pitched
        self.init = None if init is None else np.ascontiguousarray(init, dtype=np.float64)


def _device(rows, cols, width, dtype, pad_bits, data):
    import torch
    it, ft = (torch.int64, torch.float64) if dtype == np.float64 else (torch.int32, torch.float32)
    t = torch.full((rows + 1, width), pad_bits, dtype=it, device='cuda').view(ft)
    if data is not None:
        t[:rows, :cols] = torch.from_numpy(data).cuda()
    return t


def _first_diff(a, b):
    idx = np.argwhere(a != b)
    return None if len(idx) == 0 else tuple(int(i) for i in idx[0])


def guarded(ncell, launch, arrays):
    """
    Runs `launch(ld, dev)` (dev: name -> cuda tensor of `arrays`, returns the C status) at the three pitches, with
    poisoned and with zero padding.  Returns name -> [rows, cols] float64 result of every Out.
    """
    import torch
    from xanthos_b200 import _cuda as C
    runs = []
    for ld in (ncell, C.padded_ld(ncell), C.padded_ld(ncell) + 16):
        for dirty in (True, False):
            dev = {}
            for k, a in arrays.items():
                if isinstance(a, In):
                    pad = (NAN_BITS if a.a.dtype == np.float64 else F32_NAN_BITS) if dirty else 0
                    dev[k] = _device(a.rows, a.cols, ld if a.pitched else a.cols, a.a.dtype, pad, a.a)
                else:
                    dev[k] = _device(a.rows, a.cols, ld if a.pitched else a.cols, np.float64,
                                     GUARD_BITS if dirty else 0, a.init)
            C.check(launch(ld, dev))
            torch.cuda.synchronize()
            res = {}
            for k, a in arrays.items():
                if isinstance(a, Out):
                    bits = dev[k].view(torch.int64).cpu().numpy()
                    pad = np.ones(bits.shape, dtype=bool)
                    pad[:a.rows, :a.cols] = False
                    want = GUARD_BITS if dirty else 0
                    assert (bits[pad] == want).all(), "{}: padding written (ld={}, dirty={}) at {}".format(
                        k, ld, dirty, tuple(int(i) for i in np.argwhere(pad & (bits != want))[0]))
                    res[k] = bits[:a.rows, :a.cols].copy()
            runs.append((ld, dirty, res))
    ld0, _, first = runs[0]
    for ld, dirty, res in runs[1:]:
        for k in res:
            assert np.array_equal(res[k], first[k]), "{}: ld={} dirty={} differs from ld={} poisoned at {}".format(
                k, ld, dirty, ld0, _first_diff(res[k], first[k]))
    return {k: v.view(np.float64) for k, v in first.items()}


def _ptr(t):
    from xanthos_b200 import _cuda as C
    return C.ptr(t)


def _p(dev, k):
    return _ptr(dev.get(k))


def _stream():
    from xanthos_b200 import _cuda as C
    return C.stream_ptr()


def _lib():
    from xanthos_b200 import _cuda as C
    return C.lib()


def _assert_close(got, want, tol, floor=1e-6, what=''):
    with np.errstate(invalid='ignore'):
        err = max_rel(got, want, floor=floor)
    assert err < tol, (what, err)


def _assert_zero_nan_pattern(got, want, what=''):
    assert np.array_equal(np.isnan(got), np.isnan(want)), (what, 'NaN pattern')
    assert np.array_equal(got == 0, want == 0), (what, 'zero pattern', _first_diff(got == 0, want == 0))


def _assert_bits(got, want, what='', nan_bits=True):
    """Bit for bit (so -0.0 != 0.0).  nan_bits=False compares a NaN as NaN: the sign and payload of a NaN that
    arithmetic produces differ between the GPU and x86 (numpy's 0/0 is 0xfff8..., a negative NaN)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    if not nan_bits:
        got, want = np.where(np.isnan(got), np.nan, got), np.where(np.isnan(want), np.nan, want)
    g = np.ascontiguousarray(got).view(np.int64)
    w = np.ascontiguousarray(want).view(np.int64)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    assert np.array_equal(g, w), (what, _first_diff(g, w))


# ---- PET: Hargreaves-Samani -------------------------------------------------------------------------------------------

HS_LATS = (90.0, -90.0, 66.56, -66.56, 66.57, -66.57, 0.0)


@pytest.mark.parametrize("ncell,sy,ey", [(127, 1999, 1999), (257, 1999, 1999), (129, 2096, 2104), (255, 2096, 2104),
                                         (33, 1950, 2100)])
def test_hs_pet_edges(ncell, sy, ey):
    """Poles and both sides of the polar circles (the clamp of the sunset angle), tas of 0 / -0 / negative / NaN,
    tmax < tmin; one year, and 2096-2104 around the non-leap 2100."""
    from oracle import pet as opet
    rng = np.random.default_rng(ncell + sy)
    m = (ey - sy + 1) * 12
    lat = rng.uniform(-89.0, 89.0, ncell)
    lat[:len(HS_LATS)] = HS_LATS
    tas = rng.uniform(-10.0, 35.0, (ncell, m))
    tmax = tas + rng.uniform(0.0, 8.0, (ncell, m))
    tmin = tas - rng.uniform(0.0, 8.0, (ncell, m))
    swap = rng.random((ncell, m)) < 0.2
    tmax[swap], tmin[swap] = tmin[swap], tmax[swap].copy()
    for j, v in enumerate((0.0, -0.0, -3.0, np.nan)):
        tas[:, j::12][:, ::2] = v                                   # every cell, every other year
    tas.ravel()[rng.choice(ncell * m, ncell, replace=False)] = np.nan

    def launch(ld, d):
        return _lib().xan_hs_pet(_p(d, 'tas'), _p(d, 'tmax'), _p(d, 'tmin'), _p(d, 'lat'), _p(d, 'pet'), ncell, m, ld,
                                 sy, _stream())
    got = guarded(ncell, launch, dict(tas=In(tas.T), tmax=In(tmax.T), tmin=In(tmin.T), lat=In(lat[None], False),
                                      pet=Out(m, ncell)))['pet'].T
    with np.errstate(invalid='ignore'):
        want = opet.hs_pet(tas, tmax, tmin, lat, sy, ey)
    _assert_close(got, want, RTOL)
    _assert_zero_nan_pattern(got, want)
    pole = got[:2][~np.isnan(got[:2])]
    assert (pole == 0).all()                    # the reference clamps both polar day and polar night to acs = 0


# ---- PET: Thornthwaite ------------------------------------------------------------------------------------------------

def _tw_lats(rng, ncell):
    lat = rng.uniform(-1.5, 1.5, ncell)
    k = min(3, ncell)
    lat[:k] = (np.pi / 2, -np.pi / 2, 0.0)[:k]
    return lat


@pytest.mark.parametrize("nyears,sy", [(1, 1999), (2, 2099), (11, 1996), (12, 1996), (13, 1996), (95, 2010)])
def test_thornthwaite_pet_edges(nyears, sy):
    """nyears around 12 for the np.repeat day-length tiling (column k -> month k // nyears), a year of only negative or
    NaN temperatures (heat index 0), the poles; 95 years include the non-leap 2100."""
    from oracle import pet as opet
    ncell = 33 if nyears == 95 else 257
    rng = np.random.default_rng(nyears)
    ey = sy + nyears - 1
    m = nyears * 12
    lat = _tw_lats(rng, ncell)
    tas = rng.uniform(-5.0, 30.0, (ncell, m))
    tas.ravel()[rng.choice(ncell * m, max(1, ncell * m // 50), replace=False)] = np.nan
    tas.ravel()[rng.choice(ncell * m, max(1, ncell * m // 50), replace=False)] = -2.0
    y = nyears - 1
    tas[3:9, 12 * y:12 * y + 12] = -1.0                             # last year all negative ...
    tas[5:9, 12 * y:12 * y + 12:2] = np.nan                         # ... or NaN
    tas[0:3, 0:12] = -0.5                                           # and at the poles / equator in the first

    def launch(ld, d):
        return _lib().xan_thornthwaite_pet(_p(d, 'tas'), _p(d, 'lat'), _p(d, 'pet'), ncell, m, ld, sy, _stream())
    got = guarded(ncell, launch, dict(tas=In(tas.T), lat=In(lat[None], False), pet=Out(m, ncell)))['pet'].T
    with np.errstate(invalid='ignore', divide='ignore'):
        want = opet.thornthwaite_pet(tas, lat, sy, ey)
    _assert_close(got, want, RTOL)
    _assert_zero_nan_pattern(got, want)
    assert (got[5:9, 12 * y:] == 0).all()


@pytest.mark.parametrize("ncell", [1, 127, 129])
def test_thornthwaite_daylight_edges(ncell):
    from oracle import pet as opet
    from oracle.calendar_utils import MONTHDAYS, LEAP_MONTHDAYS
    lat = _tw_lats(np.random.default_rng(ncell), ncell)

    def launch(ld, d):
        return _lib().xan_thornthwaite_daylight(_p(d, 'lat'), _p(d, 'hours'), ncell, _stream())
    got = guarded(ncell, launch, dict(lat=In(lat[None], False), hours=Out(24, ncell, pitched=False)))['hours']
    want = np.concatenate([opet.daylight_hours(MONTHDAYS, lat).T, opet.daylight_hours(LEAP_MONTHDAYS, lat).T])
    _assert_close(got, want, RTOL)
    _assert_zero_nan_pattern(got, want)


# ---- PET: Hargreaves (step-wise path) ---------------------------------------------------------------------------------

@pytest.mark.parametrize("ncell,nmonths", [(257, 1), (31, 13), (255, 13)])
def test_hargreaves_pet_edges(ncell, nmonths):
    """Poles, negative and NaN dtr, NaN temperature; a single month and a month past a whole year."""
    from oracle import stepwise as ost
    from oracle.calendar_utils import set_month_arrays
    rng = np.random.default_rng(ncell * 100 + nmonths)
    ymd = set_month_arrays(24, 2000, 2001)[:nmonths]
    sd, dr = ost.calc_sinusoidal_factor(ymd)
    days = ymd[:, 2].astype(np.int32)
    lat = _tw_lats(rng, ncell)
    temp = rng.uniform(-20.0, 35.0, (ncell, nmonths))
    dtr = rng.uniform(-4.0, 16.0, (ncell, nmonths))
    dtr.ravel()[rng.choice(ncell * nmonths, max(1, ncell * nmonths // 10), replace=False)] = np.nan
    temp.ravel()[rng.choice(ncell * nmonths, max(1, ncell * nmonths // 10), replace=False)] = np.nan
    dtr[:3, 0] = (-1.0, np.nan, 5.0)
    from xanthos_b200 import _cuda as C
    sda, sdp = C.as_c(sd, np.float64)
    dra, drp = C.as_c(dr, np.float64)
    dya, dyp = C.as_c(days, np.int32)

    def launch(ld, d):
        return _lib().xan_hargreaves_pet(_p(d, 'temp'), _p(d, 'dtr'), _p(d, 'lat'), sdp, drp, dyp, _p(d, 'pet'), ncell,
                                         nmonths, ld, _stream())
    got = guarded(ncell, launch, dict(temp=In(temp.T), dtr=In(dtr.T), lat=In(lat[None], False),
                                      pet=Out(nmonths, ncell)))['pet'].T
    t, dd = np.nan_to_num(temp), np.nan_to_num(dtr)
    want = np.stack([ost.hargreaves_pet(t[:, k], dd[:, k], lat, sd[k], dr[k], days[k]) for k in range(nmonths)], axis=1)
    _assert_close(got, want, RTOL)
    _assert_zero_nan_pattern(got, want)


# ---- PET: Penman-Monteith ---------------------------------------------------------------------------------------------

PM_SY, PM_EY = 1999, 2004                # 2000 is a leap year
PM_LC_YEARS = [2000, 2003]               # land cover starts after the first model year and changes in 2003
RH_EDGES = (0.0, 69.999999, 70.0, 79.99999999, 80.0, 90.0, 95.0, 99.9999, 99.99995, 100.0)


def _pm_case(ncell, nlcs, water_idx, snow_idx, prev, seed):
    """Inputs in the oracle's layout.  Classes 1, 2, 3, 5 (never water or snow here) carry the table edges:
    laimin == laimax (fcd == 0), LAI == 0 all year, Tminopen == Tminclose, VPDopen == VPDclose."""
    rng = np.random.default_rng(seed)
    m = (PM_EY - PM_SY + 1) * 12
    T = rng.uniform(-25.0, 38.0, (ncell, m))
    d = dict(tair_load=T, TMIN_load=T - rng.uniform(0.0, 8.0, (ncell, m)), rhs_load=rng.uniform(5.0, 100.0, (ncell, m)),
             wind_load=rng.uniform(0.0, 8.0, (ncell, m)), rsds_load=rng.uniform(0.0, 350.0, (ncell, m)),
             rlds_load=rng.uniform(150.0, 450.0, (ncell, m)))
    k = max(1, ncell * m // 40)
    pos = rng.choice(ncell * m, (len(RH_EDGES), k), replace=False)
    for v, p in zip(RH_EDGES, pos):
        d['rhs_load'].ravel()[p] = v
    t = dict(cL=rng.uniform(0.001, 0.01, nlcs), beta=rng.uniform(100.0, 300.0, nlcs),
             rslimit=rng.uniform(1000.0, 5000.0, nlcs), Tminopen=rng.uniform(8.0, 12.0, nlcs),
             Tminclose=rng.uniform(-8.0, -6.0, nlcs), VPDclose=rng.uniform(28.0, 45.0, nlcs),
             VPDopen=rng.uniform(6.0, 10.0, nlcs), RBLmin=rng.uniform(55.0, 70.0, nlcs),
             RBLmax=rng.uniform(90.0, 100.0, nlcs), rc=rng.uniform(0.005, 0.02, nlcs),
             emiss=rng.uniform(0.9, 0.99, nlcs), alpha=rng.uniform(0.05, 0.4, (nlcs, 12)))
    lai = rng.uniform(0.0, 6.0, (nlcs, 12))
    lai[rng.integers(0, nlcs, 6), rng.integers(0, 12, 6)] = 0.0
    lai[1] = 2.5                                                        # laimin == laimax: fcd == 0
    lai[2] = 0.0                                                        # bare class
    t['lai'] = lai
    t['laimin'] = np.repeat(lai.min(axis=1, keepdims=True), 12, axis=1)
    t['laimax'] = np.repeat(lai.max(axis=1, keepdims=True), 12, axis=1)
    t['Tminopen'][3] = t['Tminclose'][3] = 1.5                          # Tminopen == Tminclose
    t['VPDopen'][5] = t['VPDclose'][5] = 12.0                           # VPDopen == VPDclose
    tn = d['TMIN_load']                                                 # minimum temperature on the thresholds
    tn.ravel()[rng.choice(ncell * m, k, replace=False)] = 1.5
    tn.ravel()[rng.choice(ncell * m, k, replace=False)] = t['Tminopen'][1]
    tn.ravel()[rng.choice(ncell * m, k, replace=False)] = t['Tminclose'][1]
    nly = len(PM_LC_YEARS)
    lct = np.swapaxes(rng.dirichlet(np.ones(nlcs), size=(ncell, nly)) * 100.0, 1, 2).copy()   # [N, nlcs, years]
    lct[0, :, 0] = 0.0                                                  # land-cover total 0 in one slice
    lct[1, :, :] = 0.0                                                  # ... and in all of them
    lct[2, :, 1] = 0.0
    lct[2, water_idx, 1] = 100.0                                        # all water
    lct[3, :, :] = 0.0
    lct[3, snow_idx, :] = 100.0                                         # all snow
    d.update(t, lct_load=lct, elev=rng.uniform(0.0, 3000.0, ncell))
    d['elev'][0] = 0.0
    if prev:
        pidx = rng.integers(-1, ncell, ncell).astype(np.int32)
        pidx[:3] = -1
        tp = np.where((pidx >= 0)[:, None], T[np.maximum(pidx, 0)], 0.0)
    else:
        pidx = None
        tp = np.zeros_like(T)
        tp[1:] = T[:-1]
    d['tairprev_load'] = tp
    return d, pidx


@pytest.mark.parametrize("prev", [True, False], ids=['prev_idx', 'prev_null'])
@pytest.mark.parametrize("nlcs,water_idx,snow_idx", [(7, 0, 6), (7, 4, 4), (32, 0, 6)])
@pytest.mark.parametrize("exact", ["1", "0"])
def test_pm_pet_edges(exact, nlcs, water_idx, snow_idx, prev, monkeypatch):
    """Humidity on and around the fwet / rh thresholds, LAI == 0, fcd == 0, Tminopen == Tminclose, VPDopen == VPDclose,
    land-cover totals of 0, water_idx == snow_idx, 7 and 32 classes, land cover that starts after the first model year and
    changes during the run, prev_idx given and NULL (cell 0 then reads Tp = 0)."""
    import torch
    from xanthos_b200 import _cuda as C
    from oracle import pet as opet
    monkeypatch.setenv('XANTHOS_PM_EXACT', exact)
    ncell = 129
    d, pidx = _pm_case(ncell, nlcs, water_idx, snow_idx, prev, seed=nlcs * 10 + water_idx + 2 * prev)
    m = (PM_EY - PM_SY + 1) * 12
    nly = len(PM_LC_YEARS)
    keep = []
    tabs = C.PmTables()
    tabs.nlcs, tabs.water_idx, tabs.snow_idx = nlcs, water_idx, snow_idx
    for k in ('cL', 'beta', 'rslimit', 'Tminopen', 'Tminclose', 'VPDclose', 'VPDopen', 'RBLmin', 'RBLmax', 'rc', 'emiss',
              'alpha', 'lai', 'laimin', 'laimax'):
        a, p = C.as_c(d[k], np.float64)
        keep.append(a)
        setattr(tabs, k, p)
    lc_idx = [opet.pm_land_cover_year(y, PM_LC_YEARS) for y in range(PM_SY, PM_EY + 1)]
    assert lc_idx[0] == 0 and lc_idx[-1] == 1
    lca, lcp = C.as_c(lc_idx, np.int32)
    d_pidx = None if pidx is None else torch.from_numpy(pidx).cuda()
    lct_dev = np.transpose(d['lct_load'], (2, 1, 0)).reshape(nly * nlcs, ncell)     # [year][class][cell]
    forcing = ('tair_load', 'TMIN_load', 'rhs_load', 'wind_load', 'rsds_load', 'rlds_load')

    def launch(ld, dv):
        return _lib().xan_pm_pet(*[_p(dv, k) for k in forcing], _p(dv, 'lct'), _p(dv, 'elev'), C.ptr(d_pidx),
                                 ctypes.byref(tabs), lcp, _p(dv, 'pet'), ncell, m, ld, PM_SY, _stream())
    arrays = {k: In(d[k].T) for k in forcing}
    arrays.update(lct=In(lct_dev), elev=In(d['elev'][None], False), pet=Out(m, ncell))
    got = guarded(ncell, launch, arrays)['pet'].T
    with np.errstate(all='ignore'):
        want = opet.pm_pet(d, ncell, nlcs, PM_SY, PM_EY, water_idx, snow_idx, PM_LC_YEARS)
    _assert_close(got, want, 1e-12 if exact == "1" else 1e-11)
    assert (got[1] == 0).all() and not np.isnan(got).any()


# ---- runoff: ABCD -----------------------------------------------------------------------------------------------------

def _abcd_pars(rng, n):
    lb = 1e-4
    return np.stack([rng.uniform(lb, 1 - lb, n), rng.uniform(lb, 8 - lb, n), rng.uniform(lb, 1 - lb, n),
                     rng.uniform(lb, 1 - lb, n), rng.uniform(lb, 1 - lb, n)], axis=1)


def _abcd_forcing(rng, ncell, nmonths, zero_pet):
    precip = np.abs(rng.normal(80.0, 60.0, (ncell, nmonths)))
    precip.ravel()[rng.choice(ncell * nmonths, max(1, ncell * nmonths // 500), replace=False)] = np.nan
    pet = np.zeros((ncell, nmonths)) if zero_pet else np.abs(rng.normal(90.0, 50.0, (ncell, nmonths)))
    tmin = rng.uniform(-8.0, 10.0, (ncell, nmonths))
    for v in (2.5, 0.6, np.nan):                                    # the rain / snow thresholds, and no temperature
        tmin.ravel()[rng.choice(ncell * nmonths, max(1, ncell * nmonths // 100), replace=False)] = v
    return pet, precip, tmin


def _abcd_run(basin_idx, n_basins, pars, pet, precip, tmin, nmonths, spinup):
    """xan_abcd_run on a plan made from `basin_idx` (0-based rows, -1 = not simulated) -> aet, q, sav [ncell, nmonths]."""
    import torch
    from xanthos_b200 import _cuda as C
    ncell = len(basin_idx)
    bi, bip = C.as_c(basin_idx, np.int32)
    plan = C.check_ptr(C.lib().xan_abcd_plan_create(bip, ncell, n_basins))
    try:
        d_pars = torch.from_numpy(np.ascontiguousarray(pars)).cuda()

        def launch(ld, d):
            return C.lib().xan_abcd_run(plan, _p(d, 'pet'), _p(d, 'precip'), _p(d, 'tmin'), C.ptr(d_pars), nmonths,
                                        spinup, ld, _p(d, 'aet'), _p(d, 'q'), _p(d, 'sav'), _stream())
        arrays = dict(pet=In(pet.T), precip=In(precip.T), aet=Out(nmonths, ncell), q=Out(nmonths, ncell),
                      sav=Out(nmonths, ncell))
        if tmin is not None:
            arrays['tmin'] = In(tmin.T)
        r = guarded(ncell, launch, arrays)
    finally:
        C.lib().xan_abcd_plan_destroy(plan)
    return r['aet'].T, r['q'].T, r['sav'].T


@pytest.mark.parametrize("snow", [True, False], ids=['snow', 'nosnow'])
@pytest.mark.parametrize("spinup", [25, 26, 27, 28, None], ids=['spin25', 'spin26', 'spin27', 'spin28', 'spin_all'])
@pytest.mark.parametrize("nmonths", [29, 30, 31])
def test_abcd_single_cell_basins_bitwise(nmonths, spinup, snow):
    """Month counts that leave 1, 2 or 3 months of the last 4-month stage, spin-ups that put the December segment
    boundaries on every position of a stage (25: the first segment is month 0 alone), a cell whose forcing is all NaN
    (nanmean 0 / 0) and cells not simulated (basin index -1): with zero PET and one cell per basin the run is the
    oracle's bit for bit, the cells outside come back NaN."""
    from oracle import abcd as oabcd
    spinup = nmonths if spinup is None else spinup
    ncell = 129
    rng = np.random.default_rng(nmonths * 100 + spinup)
    pet, precip, tmin = _abcd_forcing(rng, ncell, nmonths, zero_pet=True)
    precip[7] = np.nan
    pars = _abcd_pars(rng, ncell)
    basin_idx = np.arange(ncell)
    out = np.array([3, 64, 127, 128])
    basin_idx[out] = -1
    live = basin_idx >= 0
    got = _abcd_run(basin_idx, ncell, pars, pet, precip, tmin if snow else None, nmonths, spinup)
    tm = tmin[live] if snow else None
    with np.errstate(all='ignore'):
        want = oabcd.abcd_emulate(pars[live], pet[live], precip[live], tm, np.arange(live.sum()), nmonths, spinup)[:3]
    for name, g, w in zip(('aet', 'q', 'sav'), got, want):
        assert np.isnan(g[out]).all(), name
        _assert_bits(g[live], w, name, nan_bits=False)
    assert np.isnan(got[1][7]).all()


@pytest.mark.parametrize("snow", [True, False], ids=['snow', 'nosnow'])
@pytest.mark.parametrize("nmonths,spinup", [(31, 25), (30, 30), (1141, 1141)])
def test_abcd_basins_of_several_cells(nmonths, spinup, snow):
    """Basins of 1 and 33 cells (interleaved), one basin whose forcing is all NaN, cells with basin index -1; the
    re-initialisation's block reduction does not add in numpy's order, so 1e-9.  1141 months is the long case."""
    from oracle import abcd as oabcd
    rng = np.random.default_rng(nmonths + spinup)
    sizes = (1, 33, 33, 1, 5)
    ids = np.concatenate([np.full(s, b) for b, s in enumerate(sizes)] + [np.full(3, -1)])
    basin_idx = rng.permutation(ids)
    ncell = len(basin_idx)
    pet, precip, tmin = _abcd_forcing(rng, ncell, nmonths, zero_pet=False)
    precip[basin_idx == 3] = np.nan                                 # a basin without forcing
    pars = _abcd_pars(rng, len(sizes))
    live = basin_idx >= 0
    got = _abcd_run(basin_idx, len(sizes), pars, pet, precip, tmin if snow else None, nmonths, spinup)
    tm = tmin[live] if snow else None
    with np.errstate(all='ignore'):
        want = oabcd.abcd_emulate(pars[basin_idx[live]], pet[live], precip[live], tm, basin_idx[live], nmonths,
                                  spinup)[:3]
    for name, g, w in zip(('aet', 'q', 'sav'), got, want):
        assert np.isnan(g[~live]).all(), name
        _assert_close(g[live], w, RTOL, what=name)
        assert np.isnan(g[basin_idx == 3]).all(), name


def test_abcd_short_spinup_refused_before_launch():
    """Spin-up < 25 is the reference's IndexError and spin-up > nmonths a ValidationException: both refused by the host."""
    import torch
    from xanthos_b200 import _cuda as C
    bi, bip = C.as_c(np.zeros(4), np.int32)
    plan = C.check_ptr(C.lib().xan_abcd_plan_create(bip, 4, 1))
    try:
        x = torch.zeros((30, 16), dtype=torch.float64, device='cuda')
        pars = torch.full((1, 5), 0.5, dtype=torch.float64, device='cuda')
        for spin, rc in ((24, C.XAN_E_SPINUP), (31, C.XAN_E_INVALID)):
            assert C.lib().xan_abcd_run(plan, C.ptr(x), C.ptr(x), None, C.ptr(pars), 30, spin, 16, C.ptr(x), None, None,
                                        _stream()) == rc
    finally:
        C.lib().xan_abcd_plan_destroy(plan)


# ---- runoff: GWAM (step-wise path) ------------------------------------------------------------------------------------

@pytest.mark.parametrize("spinup", [0, 1, 5, None], ids=['spin0', 'spin1', 'spin5', 'spin_all'])
@pytest.mark.parametrize("nmonths", [7, 13])
def test_gwam_edges(nmonths, spinup):
    """Month counts that leave the 4-month unroll a remainder, spin-ups of 0, 1, 5 and all months, water bodies (999),
    cells without soil (0), NaN precipitation and PET; the carried soil moisture after spin-up and after the last month."""
    from oracle import stepwise as ost
    spinup = nmonths if spinup is None else spinup
    ncell = 129
    rng = np.random.default_rng(nmonths * 10 + spinup)
    pet = np.abs(rng.normal(60.0, 50.0, (ncell, nmonths)))
    precip = np.abs(rng.normal(70.0, 60.0, (ncell, nmonths)))
    precip.ravel()[rng.choice(ncell * nmonths, ncell // 4, replace=False)] = np.nan
    pet.ravel()[rng.choice(ncell * nmonths, ncell // 4, replace=False)] = np.nan
    precip[5] = np.nan
    sm_max = rng.uniform(15.0, 450.0, ncell)
    sm_max[rng.choice(ncell, 12, replace=False)] = 999.0
    sm_max[rng.choice(ncell, 6, replace=False)] = 0.0
    sm_max[[126, 127, 128]] = (999.0, 0.0, 999.0)                   # also in the last, partial block
    sm_prev = 0.5 * np.where(sm_max == 999.0, 100.0, sm_max)

    def launch(ld, d):
        return _lib().xan_gwam_run(_p(d, 'pet'), _p(d, 'precip'), _p(d, 'sm_max'), _p(d, 'sm_prev'), ncell, nmonths,
                                   spinup, ld, _p(d, 'aet'), _p(d, 'q'), _p(d, 'sav'), _p(d, 'spun'), _p(d, 'last'),
                                   _stream())
    got = guarded(ncell, launch, dict(pet=In(pet.T), precip=In(precip.T), sm_max=In(sm_max[None], False),
                                      sm_prev=In(sm_prev[None], False), aet=Out(nmonths, ncell), q=Out(nmonths, ncell),
                                      sav=Out(nmonths, ncell), spun=Out(1, ncell, pitched=False),
                                      last=Out(1, ncell, pitched=False)))
    sm = sm_prev.copy()
    with np.errstate(invalid='ignore'):
        for k in range(spinup):
            sm = ost.gwam_runoffgen(pet[:, k], precip[:, k], sm_max, sm)[2]
        want = dict(spun=sm.copy(), aet=np.zeros((ncell, nmonths)), q=np.zeros((ncell, nmonths)),
                    sav=np.zeros((ncell, nmonths)))
        for k in range(nmonths):
            want['aet'][:, k], want['q'][:, k], want['sav'][:, k] = ost.gwam_runoffgen(pet[:, k], precip[:, k], sm_max,
                                                                                       sm)
            sm = want['sav'][:, k].copy()
    want['last'] = sm
    for k in ('aet', 'q', 'sav'):
        _assert_close(got[k].T, want[k], RTOL, what=k)
        _assert_zero_nan_pattern(got[k].T, want[k], k)
    for k in ('spun', 'last'):
        _assert_close(got[k][0], want[k], RTOL, what=k)
        _assert_zero_nan_pattern(got[k][0], want[k], k)


# ---- layout ---------------------------------------------------------------------------------------------------------

F32_SPECIALS = np.array([np.nan, np.inf, -np.inf, -0.0, 1e-40, -1e-45, 1.1754942e-38, -3e-39], dtype=np.float32)


@pytest.mark.parametrize("nmonths", [1, 31, 33, 65])
@pytest.mark.parametrize("ncell", [1, 31, 33, 65])
def test_layout_transposes(ncell, nmonths):
    """NaN, +-inf, -0.0 and float32 subnormals through both transposes, with nan_to_num on and off; the float32 upload
    equals the float64 one of the same values bit for bit (float -> double is exact)."""
    from xanthos_b200 import _cuda as C
    rng = np.random.default_rng(ncell * 1000 + nmonths)
    x32 = rng.normal(0.0, 100.0, (ncell, nmonths)).astype(np.float32)
    pos = rng.choice(ncell * nmonths, max(1, ncell * nmonths // 3), replace=False)
    x32.ravel()[pos] = np.resize(np.roll(F32_SPECIALS, ncell + nmonths), len(pos))
    x64 = x32.astype(np.float64)
    x64.ravel()[pos[::5]] = np.resize(np.array([5e-324, -2.2e-308, -0.0, np.nan]), len(pos[::5]))   # float64 subnormals
    x32_wide = x32.astype(np.float64)
    for n2n in (0, 1):
        def to_mm(src, f32=False):
            fn = C.lib().xan_to_month_major_f32 if f32 else C.lib().xan_to_month_major
            return guarded(ncell, lambda ld, d: fn(_p(d, 'src'), _p(d, 'dst'), ncell, nmonths, ld, n2n, _stream()),
                           dict(src=In(src, False), dst=Out(nmonths, ncell)))['dst']
        for src in (x64, x32_wide):
            _assert_bits(to_mm(src), (np.nan_to_num(src) if n2n else src).T, ('f64', n2n))
        _assert_bits(to_mm(x32, f32=True), to_mm(x32_wide), ('f32 vs f64', n2n))

    def to_cm(ld, d):
        return C.lib().xan_to_cell_major(_p(d, 'src'), _p(d, 'dst'), ncell, nmonths, ld, _stream())
    got = guarded(ncell, to_cm, dict(src=In(x64.T), dst=Out(ncell, nmonths, pitched=False)))['dst']
    _assert_bits(got, x64, 'cell major')


# ---- aggregation ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("scaled", [True, False], ids=['scale', 'scale_null'])
@pytest.mark.parametrize("nmonths", [12, 30, 41])
def test_year_sum_scaled_bitwise(nmonths, scaled):
    """numpy.sum over 12 months times area / 1e6 (or nothing), a trailing partial year dropped (its row is not
    written: the guard row after the last year catches it)."""
    from oracle import postproc as opp
    ncell = 257
    rng = np.random.default_rng(nmonths)
    x = rng.normal(50.0, 80.0, (ncell, nmonths)) * 10.0 ** rng.integers(-3, 4, (ncell, nmonths))
    x.ravel()[rng.choice(ncell * nmonths, 20, replace=False)] = np.nan
    area = rng.uniform(1e2, 3e9, ncell)
    ny = nmonths // 12

    def launch(ld, d):
        return _lib().xan_year_sum_scaled(_p(d, 'src'), _p(d, 'scale'), ncell, nmonths, ld, _p(d, 'dst'), _stream())
    arrays = dict(src=In(x.T), dst=Out(ny, ncell))
    if scaled:
        arrays['scale'] = In((area / 1e6)[None], False)
    got = guarded(ncell, launch, arrays)['dst'].T
    want = opp.yearly_km3(x, area if scaled else np.full(ncell, 1e6))
    _assert_bits(got, want)


def test_scale_cells_in_place_bitwise():
    ncell, ntime = 257, 13
    rng = np.random.default_rng(3)
    x = rng.normal(0.0, 1e3, (ncell, ntime))
    x.ravel()[:7] = (np.nan, np.inf, -0.0, 5e-324, -np.inf, 0.0, 1e308)
    scale = rng.uniform(1e-4, 1e4, ncell)

    def launch(ld, d):
        return _lib().xan_scale_cells(_p(d, 'x'), _p(d, 'scale'), ncell, ntime, ld, _p(d, 'x'), _stream())
    got = guarded(ncell, launch, dict(x=Out(ntime, ncell, init=x.T), scale=In(scale[None], False)))['x'].T
    with np.errstate(invalid='ignore', over='ignore'):
        _assert_bits(got, x * scale[:, None])


def _groups(rng, sizes, n_out):
    """id map (1-based group ids; 0 and negative ids belong to no group) with groups of the given sizes, shuffled."""
    ids = np.concatenate([np.full(s, g + 1) for g, s in enumerate(sizes)] +
                         [np.zeros(n_out // 2, int), np.full(n_out - n_out // 2, -3)])
    return rng.permutation(ids)


def _group_table(ids, ngroups):
    cells = np.nonzero(ids > 0)[0]
    order = cells[np.argsort(ids[cells], kind='stable')].astype(np.int32)
    offsets = np.concatenate([[0], np.cumsum(np.bincount(ids[cells] - 1, minlength=ngroups))]).astype(np.int32)
    return order, offsets


GROUP_CASES = [((0, 15, 16, 17, 0, 33, 1, 32, 48), 7, 7),          # empty groups, sizes around the 16-load batch
               ((0, 15, 16, 17, 0, 33, 1, 32, 48), 7, 130),
               ((257,), 0, 129)]                                     # one group holding every cell


@pytest.mark.parametrize("sizes,n_out,ntime", GROUP_CASES, ids=['mixed-t7', 'mixed-t130', 'one-group'])
def test_group_sum_bitwise(sizes, n_out, ntime):
    import torch
    from oracle import postproc as opp
    rng = np.random.default_rng(ntime)
    ids = _groups(rng, sizes, n_out)
    ncell, ng = len(ids), len(sizes)
    x = rng.normal(10.0, 50.0, (ncell, ntime)) * 10.0 ** rng.integers(-6, 7, (ncell, ntime))   # order matters
    x.ravel()[rng.choice(ncell * ntime, ncell, replace=False)] = np.nan
    order, offsets = _group_table(ids, ng)
    d_order, d_off = torch.from_numpy(order).cuda(), torch.from_numpy(offsets).cuda()

    def launch(ld, d):
        return _lib().xan_group_sum(_p(d, 'src'), _ptr(d_order), _ptr(d_off), ng, ntime, ld, _p(d, 'out'), _stream())
    got = guarded(ncell, launch, dict(src=In(x.T), out=Out(ng, ntime, pitched=False)))['out']
    _assert_bits(got, opp.aggregation_map(ids, x))
    assert (got[[g for g, s in enumerate(sizes) if s == 0]].view(np.int64) == 0).all()


@pytest.mark.parametrize("weighted", [True, False], ids=['w', 'w_null'])
@pytest.mark.parametrize("sizes,n_out,nmonths", [((0, 15, 16, 17, 0, 33, 1, 32, 48), 7, 13),
                                                 ((0, 15, 16, 17, 0, 33, 1, 32, 48), 7, 8),
                                                 ((257,), 0, 21)], ids=['mixed-m13', 'mixed-m8', 'one-basin'])
def test_basin_sum(sizes, n_out, nmonths, weighted):
    """nansum over the basin's cells of src * w in warp-tree order against an exact sum (1e-12); an empty basin is
    0.0 exactly."""
    from xanthos_b200 import _cuda as C
    rng = np.random.default_rng(nmonths + weighted)
    ids = _groups(rng, sizes, n_out)
    ncell, nb = len(ids), len(sizes)
    basin_idx = np.where(ids > 0, ids - 1, -1)
    x = rng.uniform(0.0, 100.0, (ncell, nmonths)) * 10.0 ** rng.integers(-3, 4, (ncell, nmonths))
    x.ravel()[rng.choice(ncell * nmonths, ncell // 2, replace=False)] = np.nan
    w = rng.uniform(1e-3, 1e3, ncell) if weighted else np.ones(ncell)
    bi, bip = C.as_c(basin_idx, np.int32)
    plan = C.check_ptr(C.lib().xan_abcd_plan_create(bip, ncell, nb))
    try:
        def launch(ld, d):
            return C.lib().xan_basin_sum(plan, _p(d, 'src'), _p(d, 'w'), nmonths, ld, _p(d, 'out'), _stream())
        arrays = dict(src=In(x.T), out=Out(nmonths, nb, pitched=False))
        if weighted:
            arrays['w'] = In(w[None], False)
        got = guarded(ncell, launch, arrays)['out']
    finally:
        C.lib().xan_abcd_plan_destroy(plan)
    want = np.zeros((nmonths, nb))
    for b in range(nb):
        cells = np.nonzero(basin_idx == b)[0]
        for m in range(nmonths):
            v = x[cells, m] * w[cells]
            want[m, b] = math.fsum(v[~np.isnan(v)])
    _assert_close(got, want, 1e-12, floor=1e-300)
    empty = [b for b, s in enumerate(sizes) if s == 0]
    assert (got[:, empty].view(np.int64) == 0).all()


@pytest.mark.parametrize("ncell", [255, 257])
def test_agg_to_year_edges(ncell):
    """pandas' groupby sum / mean over 12 months (NaN skipped) at 1e-13; an all-NaN year sums to 0.0 and averages to
    NaN, exactly."""
    from oracle import postproc as opp
    nmonths = 36
    rng = np.random.default_rng(ncell)
    x = rng.normal(40.0, 30.0, (ncell, nmonths))
    x.ravel()[rng.choice(ncell * nmonths, ncell, replace=False)] = np.nan
    x[4, 12:24] = np.nan
    x[ncell - 1, 24:36] = np.nan
    for func in ('sum', 'mean'):
        def launch(ld, d):
            return _lib().xan_agg_to_year(_p(d, 'src'), _p(d, 'dst'), ncell, nmonths, ld, int(func == 'mean'), _stream())
        got = guarded(ncell, launch, dict(src=In(x.T), dst=Out(nmonths // 12, ncell)))['dst'].T
        want = opp.agg_to_year(x, func)
        _assert_close(got, want, 1e-13, what=func)
        for c, y in ((4, 1), (ncell - 1, 2)):
            if func == 'sum':
                assert np.float64(got[c, y]).view(np.int64) == 0, (c, y, got[c, y])
            else:
                assert np.isnan(got[c, y]), (c, y, got[c, y])


THRESH_CASES = [(1, 1, 129), (1, 12, 129), (2, 1, 129), (2, 12, 129), (96, 1, 129), (96, 12, 129), (97, 1, 129),
                (97, 12, 129), (1024, 1, 33), (1024, 12, 33)]


@pytest.mark.parametrize("nyear,nper,ncell", THRESH_CASES)
def test_drought_thresholds_bitwise(nyear, nper, ncell):
    """numpy.percentile 'linear' over nyear samples per (period, cell): 96 / 97 samples are both sides of the switch from
    the shared-memory to the local-memory sort, 1024 the maximum; ties, and NaN in a sample; the 10th percentile of
    getthresh and a level whose fraction takes numpy's other interpolation branch."""
    from oracle import postproc as opp
    rng = np.random.default_rng(nyear * 100 + nper)
    ntime = nyear * nper
    h = np.round(rng.normal(50.0, 20.0, (ntime, ncell)) / 4.0) * 4.0           # many ties
    h[:, :3] = 7.0                                                              # all tied
    nan_cells = rng.choice(np.arange(3, ncell), max(1, ncell // 8), replace=False)
    h[rng.integers(0, ntime, len(nan_cells)), nan_cells] = np.nan
    for q in (0.1, 0.85):
        qq = float(np.true_divide(q * 100, 100))
        prev, gamma = opp.virtual_index(nyear, qq)

        def launch(ld, d):
            return _lib().xan_drought_thresholds(_p(d, 'hist'), ncell, ntime, ld, nper, prev, gamma, _p(d, 'out'), ld,
                                                 _stream())
        got = guarded(ncell, launch, dict(hist=In(h), out=Out(nper, ncell)))['out']
        with np.errstate(invalid='ignore'):
            _assert_bits(got, opp.getthresh(h, nper, q), q)


def test_drought_thresholds_refuse_1025_samples():
    import torch
    from xanthos_b200 import _cuda as C
    assert C.DROUGHT_MAX_YEARS == 1024
    h = torch.zeros((1025 * 12, 16), dtype=torch.float64, device='cuda')
    out = torch.zeros((12, 16), dtype=torch.float64, device='cuda')
    for nper in (1, 12):
        rc = C.lib().xan_drought_thresholds(C.ptr(h), 16, 1025 * nper, 16, nper, 0, 0.5, C.ptr(out), 16, _stream())
        assert rc == C.XAN_E_INVALID and '1025' in C.lib().xan_last_error().decode()
