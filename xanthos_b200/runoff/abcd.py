"""
ABCD runoff on the B200 - drop-in for xanthos/runoff/abcd.py.

Kept from the reference: `abcd_execute` (abcd.py:394-422, the call of Components.calculate_runoff,
components.py:236-239), `abcd_parallel` (:357-391), and the `ABCD` class with `emulate()` and the
result attributes `.rsim .actual_et .soil_water_storage .pet` ([months, cells]) that the
calibration code reads (calibrate_abcd.py:153-171).  `jobs` is accepted and ignored: the basins
are not chunked over threads, every cell is one CUDA thread.
"""

import ctypes
import logging

import numpy as np

from .. import _cuda as C

_plans = {}


class BasinPlan:
    """Basin -> cells ordering on the device (xan_abcd_plan)."""

    def __init__(self, basin_idx, n_rows):
        bi, bip = C.as_c(basin_idx, np.int32)
        self.ncell = bi.shape[0]
        self.n_rows = int(n_rows)
        self.basin_idx = bi
        self._plan = C.check_ptr(C.lib().xan_abcd_plan_create(bip, self.ncell, self.n_rows))

    def __del__(self):
        try:
            if getattr(self, '_plan', None):
                C.lib().xan_abcd_plan_destroy(self._plan)
                self._plan = None
        except Exception:
            pass


def basin_plan(basin_idx, n_rows):
    """Cached plan (keyed on the content of the basin map)."""
    bi = np.ascontiguousarray(basin_idx, dtype=np.int32)
    key = (hash(bi.tobytes()), int(n_rows))
    pl = _plans.get(key)
    if pl is None:
        if len(_plans) > 16:
            _plans.clear()
        pl = _plans[key] = BasinPlan(bi, n_rows)
    return pl


def run_device(plan, pars, pet, precip, tmin, n_months, spinup_steps, want=('aet', 'q', 'sav')):
    """ABCD.emulate on device.  Returns dict of Fields."""
    torch = C.torch_cuda()
    e, p = C.as_field(pet), C.as_field(precip)
    t = None if tmin is None else C.as_field(tmin)
    n_months = int(n_months)
    if e.nmonths < n_months or p.nmonths < n_months:
        raise C.ValidationException("ABCD forcing shorter than n_months={}".format(n_months))
    pr = torch.from_numpy(np.ascontiguousarray(pars, dtype=np.float64)).cuda() if not isinstance(pars, torch.Tensor) else pars
    if pr.shape[1] == 4:   # no-snow parameter sets (a, b, c, d)
        pr = torch.cat([pr, torch.zeros((pr.shape[0], 1), dtype=pr.dtype, device=pr.device)], dim=1).contiguous()
    out = {k: C.Field.empty(e.ncell, n_months, e.ld) for k in want}
    C.check(C.lib().xan_abcd_run(plan._plan, C.ptr(e.t), C.ptr(p.t), C.ptr(t.t if t is not None else None), C.ptr(pr),
                                 n_months, int(spinup_steps), e.ld,
                                 C.ptr(out['aet'].t if 'aet' in out else None),
                                 C.ptr(out['q'].t if 'q' in out else None),
                                 C.ptr(out['sav'].t if 'sav' in out else None), C.stream_ptr()))
    return out


def run_device_sets(plan, pars_sets, pet, precip, tmin, n_months, spinup_steps, want=('aet', 'q', 'sav')):
    """ABCD.emulate of every parameter table of `pars_sets` [P, n_rows, 4 or 5] over the same forcing: a list of P
    `run_device` dicts, set k bit-identical to run_device(plan, pars_sets[k], ...).  One xan_abcd_run_sets call reads
    the forcing once for up to C.ABCD_MAX_SETS tables; more tables take several calls."""
    torch = C.torch_cuda()
    e, p = C.as_field(pet), C.as_field(precip)
    t = None if tmin is None else C.as_field(tmin)
    n_months = int(n_months)
    if e.nmonths < n_months or p.nmonths < n_months:
        raise C.ValidationException("ABCD forcing shorter than n_months={}".format(n_months))
    pr = pars_sets if isinstance(pars_sets, torch.Tensor) else torch.from_numpy(np.asarray(pars_sets, dtype=np.float64))
    if pr.dim() != 3 or pr.shape[2] not in (4, 5):
        raise C.ValidationException("parameter sets must be [P, n_rows, 4 or 5], not {}".format(tuple(pr.shape)))
    pr = pr.to(device='cuda', dtype=torch.float64)
    if pr.shape[2] == 4:   # no-snow parameter sets (a, b, c, d)
        pr = torch.cat([pr, torch.zeros(pr.shape[:2] + (1,), dtype=pr.dtype, device=pr.device)], dim=2)
    pr = pr.contiguous()
    n_sets, n_rows = int(pr.shape[0]), int(pr.shape[1])
    outs = [{k: C.Field.empty(e.ncell, n_months, e.ld) for k in want} for _ in range(n_sets)]
    for s0 in range(0, n_sets, C.ABCD_MAX_SETS):
        grp = outs[s0:s0 + C.ABCD_MAX_SETS]
        ptrs = {k: (ctypes.c_void_p * len(grp))(*[o[k].t.data_ptr() for o in grp]) if k in want else None
                for k in ('aet', 'q', 'sav')}
        C.check(C.lib().xan_abcd_run_sets(plan._plan, len(grp), n_rows, C.ptr(e.t), C.ptr(p.t),
                                          C.ptr(t.t if t is not None else None), C.ptr(pr[s0]), n_months,
                                          int(spinup_steps), e.ld, ptrs['aet'], ptrs['q'], ptrs['sav'], C.stream_ptr()))
    return outs


def _basin_rows(n_basins, basin_ids, n_rows):
    """Row of the parameter table per cell, -1 for cells outside min_id .. min_id + n_basins - 1 (abcd.py:369-389)."""
    ids = np.asarray(basin_ids).astype(np.int64)
    lo = ids.min()
    rows = ids - 1                                             # pars_abcdm[basin_ids - 1], abcd.py:332
    rows = np.where(rows < 0, rows + n_rows, rows)
    live = (ids >= lo) & (ids < lo + int(n_basins))
    if np.any(rows[live] >= n_rows):
        raise IndexError("index {} is out of bounds for axis 0 with size {}".format(int(rows[live].max()), n_rows))
    return np.where(live, rows, -1).astype(np.int32)


def abcd_parallel(n_basins, pars, basin_ids, pet, precip, tmin, n_months, spinup_steps, jobs=-1):
    """Reference abcd.py:357-391; returns the stacked [ncell, 4 * n_months] array."""
    out = _execute(n_basins, basin_ids, pet, precip, tmin, pars, n_months, spinup_steps)
    return np.hstack(out)


def _execute(n_basins, basin_ids, pet, precip, tmin, prm, n_months, spinup_steps):
    prm = np.asarray(prm, dtype=np.float64)
    rows = _basin_rows(n_basins, basin_ids, prm.shape[0])
    logging.info("\t\tProcessing spin-up and simulation for basins {}...{}".format(int(np.min(basin_ids)), n_basins))
    plan = basin_plan(rows, prm.shape[0])
    e = C.as_field(pet)
    res = run_device(plan, prm, e, precip, tmin, n_months, spinup_steps)
    if isinstance(pet, np.ndarray) and pet.shape[1] == int(n_months) and not (rows < 0).any():
        pet_h = pet                                            # passthrough, abcd.py:352
    else:
        pet_f = C.Field(e.t[:int(n_months)], e.ncell)
        pet_h = pet_f.to_host()
        if (rows < 0).any():            # host copy differs from the device field -> it is not registered
            C.host_sync()
            pet_h[rows < 0, :] = np.nan
        else:
            pet_h = C.remember(pet_h, pet_f)
    aet = C.remember(res['aet'].to_host(), res['aet'])
    q = C.remember(res['q'].to_host(), res['q'])
    sav = C.remember(res['sav'].to_host(), res['sav'])
    return pet_h, aet, q, sav


def abcd_execute(n_basins, basin_ids, pet, precip, tmin, calib_file, n_months, spinup_steps, jobs):
    """Reference abcd.py:394-422: returns (pet, aet, q, sav), each [ncell, n_months]."""
    prm = calib_file if isinstance(calib_file, np.ndarray) else np.load(calib_file)
    return _execute(n_basins, basin_ids, pet, precip, tmin, prm, n_months, spinup_steps)


class ABCD:
    """
    Same constructor and result attributes as the reference class (abcd.py:18-311): per-cell
    parameters `pars` [n, 4 or 5], forcing [n, months], `basin_ids` [n] grouping the cells for the
    spin-up re-initialisation.  `emulate()` runs spin-up + simulation on the device.
    """

    def __init__(self, pars, pet, precip, tmin, basin_ids, process_steps, spinup_steps, method='dist'):
        self.nosnow = tmin is None
        self.pars = np.ascontiguousarray(pars, dtype=np.float64)
        self.basin_ids = np.asarray(basin_ids)
        self.steps = int(process_steps)
        self.spinup_steps = int(spinup_steps)
        self.method = method
        self._pet, self._precip, self._tmin = pet, precip, tmin
        self.pet = np.asarray(pet).T[0:self.steps, :] if not isinstance(pet, C.Field) else None
        self.rsim = self.actual_et = self.soil_water_storage = None

    def emulate(self):
        n = self.pars.shape[0]
        # per-cell parameters: every cell is its own row; the basin grouping only drives the re-init
        uniq, inv = np.unique(self.basin_ids, return_inverse=True)
        # the library keys parameters and re-init groups on the same row, so group rows must carry
        # identical parameters; fall back to one row per (group, parameter set) pair
        key = np.concatenate([inv[:, None].astype(np.float64), self.pars], axis=1)
        rows_u, rows = np.unique(key, axis=0, return_inverse=True)
        rows = rows.reshape(-1)
        if len(rows_u) != len(uniq):
            raise C.ValidationException("ABCD: cells of one basin must share one parameter set")
        plan = basin_plan(rows.astype(np.int32), len(rows_u))
        res = run_device(plan, rows_u[:, 1:], self._pet, self._precip, self._tmin, self.steps, self.spinup_steps)
        self.actual_et = res['aet'].t[:, :n].cpu().numpy()
        self.rsim = res['q'].t[:, :n].cpu().numpy()
        self.soil_water_storage = res['sav'].t[:, :n].cpu().numpy()

    def spinup(self):
        raise NotImplementedError("spin-up and simulation are fused on the device; call emulate()")

    simulate = spinup
