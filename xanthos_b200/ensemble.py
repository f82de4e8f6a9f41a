"""
Multi-member runs of the hot path (BASELINE.json config 5: "64-member ESM x SSP scenario ensemble ... sharded by member").

The reference has no ensemble driver: a user loops over configuration files, one `Xanthos(ini).execute()` per scenario
(xanthos/model.py, components.py:298-385), and every scenario re-reads the static data.  Here the static part (land
cover, PM tables, basin plan, routing plan, ABCD parameters) is staged once and the members stream through
PET -> ABCD -> MRTM with their copies overlapped:

    h2d stream     : forcing of the next members  (8 fields each, pinned host -> HBM; transposed to month-major on the
                     compute stream)
    compute stream : transposes, PM -> ABCD of members k and k+1, then ONE routing launch for both
                     (`route_device_batch`: the thread blocks of the two members share the SMs), basin aggregates,
                     output transposes.  `XANTHOS_ENSEMBLE_FRONT=1` moves PM -> ABCD of the NEXT pair to a stream of
                     its own, beside the routing launch: measured slower (75.7 against 72.0 ms per pair - every block
                     that shares an SM with the latency-bound routing chain slows it by more than it saves), so it is off.
    d2h stream     : requested outputs of the members before  (HBM -> pinned host, cell-major like the reference's arrays)

The forcing of at most `prefetch_depth` (4 = two pairs) members is on its way ahead of the group being computed, into a
fixed ring of device staging buffers (no allocation inside the pipeline).  Only the variables named in `output_vars` are copied back (the reference
keeps PET, AET, Q, Sav, ChStorage and Avg_ChFlow of a scenario in host memory but writes `output_vars` only,
data_writer/out_writer.py:60-110).  With torch.distributed initialised the members are dealt in contiguous blocks to the ranks
(no collective in the data path) and the basin aggregates [n_members, 2, nmonths, n_basins] are gathered at the end.

An `OutputSpec` applies the reference's output options (yearly, km3, basin / country / region sums) and across-member
statistics on the device, in front of the copy back (`run_ensemble(..., spec=...)`): the copy back, not the compute, is
what limits multi-GPU runs, and a user who wants reduced output no longer pulls every monthly grid to the host.

The PET model and the routing are those of the reference's [PET] and [Routing] sections: `EnsembleStatics(pet=...)`
takes 'pm' (above), 'hs' (Hargreaves-Samani), 'thornthwaite' or 'none' (PET given with every member), and
`routing=False` stops after ABCD: each member is then uploaded, run through PET -> ABCD and copied back on its own, and
the run is bounded by the host -> device link.

`run_parameter_ensemble` runs the other ensemble, parameter uncertainty: ONE forcing and many ABCD parameter tables.  The
forcing is uploaded and its PET computed once; the tables go through ABCD several per launch (xan_abcd_run_sets reads
each forcing value once for the sets of a thread), then through routing and the output reductions exactly as members.
"""

from types import SimpleNamespace

import numpy as np

from . import _cuda as C
from . import sharding
from .pet import hargreaves_samani as hs_mod
from .pet import penman_monteith as pm_mod
from .pet import thornthwaite as th_mod
from .runoff import abcd as abcd_mod
from .routing import mrtm as mrtm_mod

PM_FORCING = ('tair_load', 'TMIN_load', 'rhs_load', 'wind_load', 'rsds_load', 'rlds_load')
FORCING = PM_FORCING + ('precip', 'tmin')
# the member fields of the PET models (pet_module of the .ini), named as DataLoader names them; ABCD adds precip, tmin
PET_FORCING = {'pm': PM_FORCING, 'hs': ('hs_tas', 'hs_tmax', 'hs_tmin'), 'thornthwaite': ('tair',), 'none': ('pet',)}
PET_MODELS = tuple(PET_FORCING)
OUTPUTS = ('pet', 'aet', 'q', 'soilmoisture', 'chstorage', 'avgchflow')
ROUTED_OUTPUTS = ('chstorage', 'avgchflow')
PM_STATICS = ('pm_tables', 'lct_load', 'elev', 'water_idx', 'snow_idx', 'lc_years', 'nlcs')
ROUTING_STATICS = ('flow_dist', 'velocity', 'upstream_matrix', 'ndays')
GROUP_SCALES = ('basin', 'country', 'region')
STATS = ('mean', 'std', 'min', 'max')
DROUGHT_VARS = ('q', 'soilmoisture')
DROUGHT_SUMMARY = ('drought_months', 'events', 'longest_duration', 'peak_severity')
DROUGHT_FIELDS = ('severity', 'intensity', 'duration')
# Parameter tables per ABCD launch of an unrouted parameter ensemble (routed groups stay pairs, the routing launch's
# unit).  B200, bench world (tools/parameter_ensemble_bench.py, DESIGN.md section 6): one xan_abcd_run_sets call takes
# 0.38 ms per set at 4 sets and 0.34 at 8, against 0.53 per single-set call; 4 keeps most of the gain with half the
# pinned output grids of 8 (3 x group per output variable).
PARAMETER_SETS_PER_LAUNCH = 4


def forcing_fields(pet):
    """The keys of an ensemble member for PET model `pet` ('pm', 'hs', 'thornthwaite' or 'none'): the PET model's
    fields, then 'precip' and 'tmin' of ABCD."""
    if pet not in PET_FORCING:
        raise C.ValidationException("unknown PET model {!r}; choose from {}".format(pet, PET_MODELS))
    return PET_FORCING[pet] + ('precip', 'tmin')


class DroughtSpec:
    """
    Drought statistics of every member, the [Drought] section of a configuration (ConfigReader.configure_drought_stats)
    applied to the member's monthly mm field of `var` ('q' or 'soilmoisture'), whatever the spec's yearly / km3 options:

      thresholds       host array [K, ncell]: the thresholds of every member (drought_thresholds of the .ini), row t % K
                       for month t; staged on the device once
      threshold_years  (start, end) when no thresholds are given: each member's thresholds are its 10th percentile per
                       period over the months DroughtStats.calculate_thresholds takes (the slice end
                       (end + 1 - start) * 12 is an index, as in the reference), with `nper` periods
      fields           also return the member's severity / intensity / duration grids [ncell, nmonths]

    Every member gets its summary per cell - drought months, events, longest duration, peak severity - and the runner
    counts per cell and month how many members are in drought (a month is dry when the field is below the threshold;
    NaN is never dry).  The severity / intensity / duration and the thresholds are bitwise DroughtStats' on the member.
    """

    def __init__(self, var='q', thresholds=None, threshold_years=None, nper=12, fields=False):
        var = str(var).lower()
        if var not in DROUGHT_VARS:
            raise C.ValidationException("drought variable must be one of {}, not {!r}".format(DROUGHT_VARS, var))
        if (thresholds is None) == (threshold_years is None):
            raise C.ValidationException("give drought thresholds or threshold_years (one of the two)")
        if int(nper) != nper or nper < 1:
            raise C.ValidationException("nper must be a positive integer, not {!r}".format(nper))
        self.var, self.nper, self.fields = var, int(nper), bool(fields)
        self.thresholds = self.threshold_years = None
        if thresholds is not None:
            th = np.array(thresholds, dtype=np.float64, order='C')      # staged as [K][ncell] rows
            if th.ndim != 2 or th.shape[0] < 1:
                raise C.ValidationException("drought thresholds must be [K, ncell] with K >= 1, not {}".format(th.shape))
            self.thresholds = th
        else:
            years = tuple(int(y) for y in threshold_years)
            if len(years) != 2:
                raise C.ValidationException("threshold_years must be (start, end), not {!r}".format(threshold_years))
            self.threshold_years = years

    def reference_months(self, start_year, end_year):
        """(first, end) of the months the per-member thresholds are computed from, in a run of start_year .. end_year
        (DroughtStats.calculate_thresholds' slice); raises ValidationException where the reference would fail."""
        sy, ey = self.threshold_years
        if sy < start_year or ey > end_year:
            raise C.ValidationException("drought threshold years {} - {} are outside the run {} - {}".format(
                sy, ey, start_year, end_year))
        nmonths = (end_year - start_year + 1) * 12
        first, end = (sy - start_year) * 12, (ey + 1 - sy) * 12
        n = len(range(nmonths)[first:end])
        if n == 0 or n % self.nper or n // self.nper > C.DROUGHT_MAX_YEARS:
            raise C.ValidationException(
                "drought reference period: months [{}:{}] of the run give {} months, not a positive multiple of {} "
                "periods of at most {} years".format(first, end, n, self.nper, C.DROUGHT_MAX_YEARS))
        return first, end

    def validate(self, ncell, start_year, end_year):
        """Refuses a spec that cannot run on ncell cells and the years start_year .. end_year."""
        if self.thresholds is not None:
            if self.thresholds.shape[1] != ncell:
                raise C.ValidationException("drought thresholds have {} cells, the run {}".format(
                    self.thresholds.shape[1], ncell))
        else:
            self.reference_months(start_year, end_year)

    def __repr__(self):
        src = ('thresholds=<{} x {}>'.format(*self.thresholds.shape) if self.thresholds is not None
               else 'threshold_years={}'.format(self.threshold_years))
        return 'DroughtSpec(var={!r}, {}, nper={}, fields={})'.format(self.var, src, self.nper, self.fields)


class OutputSpec:
    """
    What the ensemble runner computes from each member's monthly outputs on the device before anything is copied back:

      output_in_year  yearly sum (mean for avgchflow) of every variable, NaN skipped (OutWriter.write, out_writer.py:103-112)
      output_unit     'mm' or 'km3': mm -> km3 by `area / 1e6` after the yearly aggregation, never for avgchflow
                      (out_writer.py:114-115)
      group_sums      subset of ('basin', 'country', 'region'): sums of q after its conversion over the cells of every
                      id > 0, in cell-index order, NaN skipped, [max(ids), ntime] (OutWriter.write_aggregates,
                      out_writer.py:250-265)
      member_fields   False: no per-member grid is copied back (group sums and statistics only)
      stats           subset of ('mean', 'std', 'min', 'max') over the members, per (cell, time step) of every output
                      variable; std with `ddof` like numpy.std
      quantiles       levels in [0, 1], in the order given: numpy.quantile(members, levels, axis=0) (method 'linear')
                      per (cell, time step) of every output variable; the median is quantiles=(0.5,)
      drought         DroughtSpec: drought statistics of every member and the across-member drought frequency

    Every member's grids and group sums are bit-identical to what OutWriter.write / write_aggregates produce from that
    member's monthly outputs.  chstorage is never written through OutWriter: it is rejected with yearly or km3 output.
    """

    def __init__(self, output_in_year=False, output_unit='mm', group_sums=(), member_fields=True, stats=(), ddof=0,
                 quantiles=(), drought=None):
        if output_unit not in ('mm', 'km3'):
            raise C.ValidationException("output_unit must be 'mm' or 'km3', not {!r}".format(output_unit))
        group_sums, stats = tuple(group_sums), tuple(stats)
        bad = [g for g in group_sums if g not in GROUP_SCALES] + [s for s in stats if s not in STATS]
        if bad or len(set(group_sums)) != len(group_sums) or len(set(stats)) != len(stats):
            raise C.ValidationException("unknown or repeated group sums / statistics {} (choose from {} and {})".format(
                list(group_sums) + list(stats), GROUP_SCALES, STATS))
        if int(ddof) != ddof or ddof < 0:
            raise C.ValidationException("ddof must be a non-negative integer, not {!r}".format(ddof))
        quantiles = tuple(float(q) for q in quantiles)
        if (not all(0.0 <= q <= 1.0 for q in quantiles) or len(set(quantiles)) != len(quantiles)
                or len(quantiles) > C.ENS_MAX_LEVELS):
            raise C.ValidationException("quantile levels must be distinct, in [0, 1] and at most {}, not {}".format(
                C.ENS_MAX_LEVELS, quantiles))
        if drought is not None and not isinstance(drought, DroughtSpec):
            raise C.ValidationException("drought must be a DroughtSpec, not {!r}".format(drought))
        self.quantiles, self.drought = quantiles, drought
        self.output_in_year, self.output_unit = bool(output_in_year), output_unit
        self.group_sums, self.member_fields, self.stats, self.ddof = group_sums, bool(member_fields), stats, int(ddof)

    @classmethod
    def from_settings(cls, settings, member_fields=True, stats=(), ddof=0, quantiles=(), drought=False):
        """The output options of a parsed configuration (data_reader.ini_reader.ConfigReader): OutputInYear,
        OutputUnit and the AggregateRunoffBasin / Country / GCAMRegion flags; with drought=True also its [Drought]
        section (drought_var, and drought_thresholds loaded with np.load or the threshold years and nper)."""
        unit = int(settings.OutputUnit)
        if unit not in (0, 1):
            raise C.ValidationException("OutputUnit must be 0 (mm) or 1 (km3), not {}".format(unit))
        dspec = None
        if drought:
            if getattr(settings, 'drought_var', None) is None:
                raise C.ValidationException("drought output requested, but the configuration has no [Drought] section "
                                            "(CalculateDroughtStats = 1)")
            if settings.drought_thresholds is not None:
                dspec = DroughtSpec(settings.drought_var, thresholds=np.load(settings.drought_thresholds))
            else:
                dspec = DroughtSpec(settings.drought_var, nper=settings.threshold_nper,
                                    threshold_years=(settings.threshold_start_year, settings.threshold_end_year))
        flags = (settings.AggregateRunoffBasin, settings.AggregateRunoffCountry, settings.AggregateRunoffGCAMRegion)
        return cls(output_in_year=bool(int(settings.OutputInYear)), output_unit=('mm', 'km3')[unit],
                   group_sums=tuple(g for g, f in zip(GROUP_SCALES, flags) if int(f)), member_fields=member_fields,
                   stats=stats, ddof=ddof, quantiles=quantiles, drought=dspec)

    def __repr__(self):
        return ('OutputSpec(output_in_year={}, output_unit={!r}, group_sums={}, member_fields={}, stats={}, ddof={}, '
                'quantiles={}{})'.format(self.output_in_year, self.output_unit, self.group_sums, self.member_fields,
                                         self.stats, self.ddof, self.quantiles,
                                         '' if self.drought is None else ', drought={!r}'.format(self.drought)))


def parameter_sets(parameter_sets, n_rows):
    """
    ABCD parameter tables as float64 [P, n_rows, 5] (host only): `parameter_sets` is one [P, n_rows, 4 or 5] array or a
    sequence of [n_rows, 4 or 5] tables (a, b, c, d[, m]; a 4-column table gets m = 0, no snow melt, as run_device
    gives it).  Raises ValidationException for a table with another row count, another column count or another rank.
    """
    if hasattr(parameter_sets, 'ndim'):
        a = np.asarray(parameter_sets, dtype=np.float64)
        if a.ndim != 3:
            raise C.ValidationException("parameter sets must be one [P, n_rows, 4 or 5] array or a sequence of "
                                        "[n_rows, 4 or 5] tables, not an array of shape {}".format(a.shape))
        tables = list(a)
    else:
        tables = [np.asarray(t, dtype=np.float64) for t in parameter_sets]
    if not tables:
        raise C.ValidationException("no parameter set given")
    out = np.zeros((len(tables), int(n_rows), 5), dtype=np.float64)
    for k, t in enumerate(tables):
        if t.ndim != 2:
            raise C.ValidationException("parameter set {} has shape {}, not [n_rows, 4 or 5]".format(k, t.shape))
        if t.shape[0] != int(n_rows):
            raise C.ValidationException("parameter set {} has {} rows, the statics' ABCD table {}".format(
                k, t.shape[0], int(n_rows)))
        if t.shape[1] not in (4, 5):
            raise C.ValidationException("parameter set {} has {} columns, not 4 (a, b, c, d) or 5 (a, b, c, d, m)".format(
                k, t.shape[1]))
        out[k, :, :t.shape[1]] = t
    return out


_parameter_sets = parameter_sets      # run_parameter_ensemble's argument of the same name hides the function


def merge_drought_counts(a, na, b, nb):
    """Drought count partial `a` (of na members) absorbs partial `b` (of nb members), in place; returns a.  The counts
    are integers, so the sum is exact in any order."""
    a[0].add_(b[0])
    return a


QUANTILE_CHUNK_BYTES = 2 << 30    # budget of the [n_members, chunk, ld] buffers that bring the members of several
                                  # runners or ranks together, all variables: enough for one time step of 256 members


def member_quantiles(stack, ncell, levels, out, t0=0):
    """
    numpy.quantile(members, levels, axis=0) (method 'linear') of a month-major member stack [n, nt, ld] (cuda float64,
    unit stride along cells; any member and time stride), written to columns t0 .. t0 + nt of the cell-major cuda
    tensor out [len(levels), ncell, ntime].  One xan_ens_quantiles launch for all levels; a member that is NaN at a
    (cell, step) makes every level NaN there.  1 <= n <= 256.
    """
    from .drought.drought_stats import virtual_index
    n, nt = int(stack.shape[0]), int(stack.shape[1])
    if not 1 <= n <= C.ENS_MAX_MEMBERS:
        raise C.ValidationException("quantiles over {} members (1 to {})".format(n, C.ENS_MAX_MEMBERS))
    if stack.stride(2) != 1 or tuple(out.shape[:2]) != (len(levels), ncell) or not out.is_contiguous():
        raise C.ValidationException("member stack {} / output {} do not fit {} levels of {} cells".format(
            tuple(stack.shape), tuple(out.shape), len(levels), ncell))
    idx = [virtual_index(n, q) for q in levels]
    lo, p_lo = C.as_c([i for i, _ in idx], np.int32)
    gamma, p_gamma = C.as_c([g for _, g in idx], np.float64)
    C.check(C.lib().xan_ens_quantiles(C.ptr(stack), stack.stride(0), n, int(ncell), stack.stride(1), int(t0),
                                      int(t0) + nt, int(out.shape[2]), len(levels), p_lo, p_gamma, C.ptr(out),
                                      C.stream_ptr()))
    return out


def lossless_float32(member, pin=True):
    """
    Returns the member with every forcing array whose values are all exactly representable in single precision replaced
    by a float32 copy (pinned when a device is present); the others are kept.  Climate-model forcing is single precision
    on disk (NetCDF float variables) and only widened to float64 by the loader (data_load.py:288-340), so the copy is
    lossless: float -> double on the device is exact and every result stays bit-identical, while the host -> device
    traffic - the limiter of multi-GPU ensemble runs - halves.  NaN (missing data) counts as representable.
    Call it once per member where the data are loaded; it costs a pass over the arrays on the host.  The forcing keys
    of every PET model are converted (those the member has); an array that is several fields of the member (tmin
    and hs_tmin read from one file) is converted once and stays one array, so it still crosses the link once.
    """
    out, done = dict(member), {}
    for k in dict.fromkeys(key for pet in PET_MODELS for key in forcing_fields(pet)):
        if k not in member:
            continue
        if id(member[k]) in done:
            out[k] = done[id(member[k])]
            continue
        a = np.asarray(member[k])
        if a.dtype == np.float64:
            a32 = a.astype(np.float32)
            back = a32.astype(np.float64)
            if np.array_equal(back, a, equal_nan=True):
                if pin and C.device_available():
                    t = C.torch_cuda().from_numpy(a32).pin_memory()
                    a32 = t.numpy()
                out[k] = a32
        done[id(member[k])] = out[k]
    return out


class EnsembleStatics:
    """
    Everything that does not change from member to member, staged on the device once.

      pet        PET model of the members, spelled as pet_module of the .ini: 'pm' (Penman-Monteith: pm_tables,
                 lct_load, elev, water_idx, snow_idx, lc_years and nlcs are required), 'hs' (Hargreaves-Samani),
                 'thornthwaite' or 'none' (every member brings its PET); other than 'pm' the PM arguments may be None
                 and are not staged.  `forcing_fields(pet)` names the member keys.
      latitude   degrees per cell (coords[:, 2]), required for 'hs' and 'thornthwaite' (in radians,
                 np.radians(latitude), as DataLoader.lat_radians)
      routing    False: no MRTM, the members stop after ABCD; flow_dist, velocity, upstream_matrix and ndays may be
                 None and dt / routing_spinup are not used

    A configuration that cannot run raises ValidationException here, naming what is missing.
    """

    def __init__(self, ncell, start_yr, end_yr, pm_tables, lct_load, elev, water_idx, snow_idx, lc_years, nlcs,
                 n_basins, basin_ids, abcd_pars, area, flow_dist, velocity, upstream_matrix, ndays, dt=3 * 3600,
                 runoff_spinup=None, routing_spinup=None, country_ids=None, region_ids=None, pet='pm', latitude=None,
                 routing=True):
        forcing_fields(pet)
        given = dict(zip(PM_STATICS + ROUTING_STATICS, (pm_tables, lct_load, elev, water_idx, snow_idx, lc_years, nlcs,
                                                        flow_dist, velocity, upstream_matrix, ndays)))
        need = (PM_STATICS if pet == 'pm' else ()) + (ROUTING_STATICS if routing else ())
        missing = [k for k in need if given[k] is None]
        if pet in ('hs', 'thornthwaite') and latitude is None:
            missing.append('latitude')
        if missing:
            raise C.ValidationException("EnsembleStatics(pet={!r}, routing={}) needs {}".format(
                pet, bool(routing), ', '.join(missing)))
        if latitude is not None and np.asarray(latitude).reshape(-1).shape[0] != int(ncell):
            raise C.ValidationException("latitude has {} entries for {} cells".format(
                np.asarray(latitude).reshape(-1).shape[0], int(ncell)))
        torch = C.torch_cuda()
        self.pet, self.routing = pet, bool(routing)
        self.ncell, self.start_yr, self.end_yr = int(ncell), int(start_yr), int(end_yr)
        self.nmonths = (self.end_yr - self.start_yr + 1) * 12
        self.ld = C.padded_ld(self.ncell)
        if pet == 'pm':
            self.tables = dict(pm_tables)
            self.water_idx, self.snow_idx = int(water_idx), int(snow_idx)
            self.lc_years, self.nlcs = list(lc_years), int(nlcs)
            self.d_lct = pm_mod.stage_land_cover(lct_load, self.ld)
            self.d_elev = C.dev_vector(elev)
        # HS takes degrees, Thornthwaite radians: np.radians of the float64 degrees, DataLoader's lat_radians bit for bit
        self.d_lat = None
        if pet in ('hs', 'thornthwaite'):
            lat = np.asarray(latitude, dtype=np.float64).reshape(-1)
            self.d_lat = C.dev_vector(lat if pet == 'hs' else np.radians(lat))
        self.n_basins = int(n_basins)
        self.basin_ids = np.asarray(basin_ids)
        rows = abcd_mod._basin_rows(self.n_basins, self.basin_ids, np.asarray(abcd_pars).shape[0])
        self.plan = abcd_mod.basin_plan(rows, self.n_basins)
        self.d_pars = torch.from_numpy(np.ascontiguousarray(abcd_pars, dtype=np.float64)).cuda()
        self.d_area = C.dev_vector(area)
        self.d_area_km3 = self.d_area * 1e-6
        self.runoff_spinup = self.nmonths if runoff_spinup is None else int(runoff_spinup)
        self.d_L = self.d_V = self.um = self.ndays = None
        if self.routing:
            self.d_L, self.d_V = C.dev_vector(flow_dist), C.dev_vector(velocity)
            self.um = upstream_matrix
            self.ndays = np.asarray(ndays, dtype=np.int32)[:self.nmonths]
        self.dt = float(dt)
        self.routing_spinup = self.nmonths if routing_spinup is None else int(routing_spinup)
        self.area = area
        self.group_ids = {'basin': self.basin_ids, 'country': country_ids, 'region': region_ids}
        self._group_tables, self._km3 = {}, None

    def group_table(self, scale):
        """Device (order, offsets, ngroups) of xan_group_sum for 'basin' / 'country' / 'region', built once."""
        hit = self._group_tables.get(scale)
        if hit is None:
            from .diagnostics.time_series import group_plan
            ids = self.group_ids.get(scale)
            if ids is None:
                raise C.ValidationException("{} group sums requested, but no {}_ids were given to EnsembleStatics".format(
                    scale, scale))
            ids = np.asarray(ids).astype(np.int64).reshape(-1)
            if ids.shape[0] != self.ncell:
                raise C.ValidationException("{}_ids has {} entries for {} cells".format(scale, ids.shape[0], self.ncell))
            order, offsets, ng = group_plan(ids)
            if ng < 1:
                raise C.ValidationException("{}_ids has no positive id".format(scale))
            torch = C.torch_cuda()
            hit = self._group_tables[scale] = (torch.from_numpy(order).cuda(), torch.from_numpy(offsets).cuda(), ng)
        return hit

    def km3_scale(self):
        """Device vector area / 1e6, OutWriter.conversion_mm_km3 (not d_area_km3 = area * 1e-6: the last bit differs)."""
        if self._km3 is None:
            self._km3 = C.dev_vector(np.asarray(self.area, dtype=np.float64).reshape(-1) / 1e6)
        return self._km3

    def data_ns(self, fields):
        d = dict(self.tables)
        d.update({k: fields[k] for k in PM_FORCING})
        d['lct_load'] = self.d_lct
        d['elev'] = self.d_elev
        return SimpleNamespace(**d)


class EnsembleRunner:
    def __init__(self, statics, output_vars=('q', 'avgchflow'), aggregates=True, prefetch_depth=4, group=None,
                 spec=None):
        torch = C.torch_cuda()
        self.prefetch_depth = max(1, int(prefetch_depth))   # members whose forcing may be on its way ahead of the compute
        if group is None:                                   # members routed by one launch; nothing to share unrouted
            group = 2 if statics.routing else 1
        self.group = max(1, int(group))
        bad = [v for v in output_vars if v not in OUTPUTS]
        if bad:
            raise C.ValidationException("unknown output variable(s) {}; choose from {}".format(bad, OUTPUTS))
        routed = [v for v in output_vars if v in ROUTED_OUTPUTS]
        if routed and not statics.routing:
            raise C.ValidationException("output variable(s) {} need routing; the statics have routing=False".format(
                routed))
        self.s, self.output_vars, self.aggregates = statics, tuple(output_vars), bool(aggregates)
        self.n_agg_rows = 2 if statics.routing else 1       # basin runoff (and the basin sum of the mean streamflow)
        self.spec = spec
        self.ntime = statics.nmonths // 12 if spec is not None and spec.output_in_year else statics.nmonths
        if spec is not None:
            if 'chstorage' in self.output_vars and (spec.output_in_year or spec.output_unit == 'km3'):
                raise C.ValidationException("chstorage has no yearly or km3 output (OutWriter never writes it)")
            self._groups = {g: statics.group_table(g) for g in spec.group_sums}
            # group sums are of q as it is written (after the yearly aggregation and the unit conversion)
            self._reduce_vars = self.output_vars + (('q',) if spec.group_sums and 'q' not in self.output_vars else ())
        self._stats_state, self.n_stats = None, 0   # across-member accumulators: var -> (sum, m2) and (min, max)
        self._stack, self.n_stacked = None, 0       # quantiles: var -> every member's reduced field [n, ntime, ld]
        self._drought = spec.drought if spec is not None else None
        self._drought_count, self.n_drought = None, 0   # members in drought per month and cell, int32 [nmonths, ld]
        if self._drought is not None:
            self._drought.validate(statics.ncell, statics.start_yr, statics.end_yr)
            self._drought_th = (None if self._drought.thresholds is None
                                else torch.from_numpy(self._drought.thresholds).cuda())
        # One pair of copy streams per process and device, not per runner: torch's caching allocator keeps freed blocks
        # per STREAM, so every new stream starts with an empty pool - a runner per run_ensemble call with fresh streams
        # left 6 - 9 GB of staging blocks cached under dead streams per call, and after a dozen calls the allocator had
        # to cudaFree them (a device-wide synchronisation) in the middle of the uploads: 250 - 450 ms per stalled upload.
        self.h2d, self.d2h = C.copy_stream('ensemble_h2d'), C.copy_stream('ensemble_d2h')
        import os as _os
        self.front = C.copy_stream('ensemble_front') if _os.environ.get('XANTHOS_ENSEMBLE_FRONT', '0') == '1' else None
        self.h2d_bytes = self.d2h_bytes = 0
        self._slots = None          # ring of device staging buffers for the uploads, depth + group slots
        self._torch = torch
        import os
        self.timeline = [] if os.environ.get('XANTHOS_ENSEMBLE_TIMELINE') else None   # per member: stage event pairs

    # ---- the three pipeline stages (everything is enqueued, nothing waits) ------------------------------------------
    def _slot_buffer(self, slot, k):
        """Device staging buffer of forcing field k in ring slot `slot` (made on first use, then reused for the whole
        run: a `cudaMalloc` per upload now and then stalls for hundreds of ms while a routing launch is running)."""
        torch = self._torch
        if self._slots is None or len(self._slots) <= slot:
            self._slots = (self._slots or []) + [dict() for _ in range(slot + 1 - len(self._slots or []))]
        b = self._slots[slot].get(k)
        if b is None:
            b = self._slots[slot][k] = torch.empty(self.s.ncell * self.s.nmonths, dtype=torch.float64, device='cuda')
        return b

    def _upload(self, member, slot):
        torch = self._torch
        if callable(member):
            member = member()
        keys = forcing_fields(self.s.pet)
        missing = [k for k in keys if k not in member]
        if missing:
            raise C.ValidationException("ensemble member lacks {} (pet={!r})".format(missing, self.s.pet))
        # an array that is several fields of the member (hs_tmin and tmin from one file) crosses the link once
        first = {}
        for k in keys:
            first.setdefault(id(member[k]), k)
        staged = {}
        # staging buffers allocated on the compute stream (its pool is reused)
        bufs = {k: self._slot_buffer(slot, k) for k in keys if first[id(member[k])] == k}
        # Only copy-engine work goes on the h2d stream.  The transposes to month-major run on the compute stream in front
        # of the member's kernels: a kernel on the h2d stream would wait for SM resources behind the routing kernel of
        # the previous member (one cooperative block per SM, the whole register file) and hold up the next copy.
        with torch.cuda.stream(self.h2d):
            e0 = self._mark(self.h2d)
            for k in keys:
                if first[id(member[k])] != k:
                    staged[k] = staged[first[id(member[k])]]
                    continue
                a = member[k]
                if tuple(a.shape) != (self.s.ncell, self.s.nmonths):
                    raise C.ValidationException("member field {} has shape {}, expected {}".format(
                        k, tuple(a.shape), (self.s.ncell, self.s.nmonths)))
                if not isinstance(a, torch.Tensor):
                    a = np.asarray(a)
                    if a.dtype not in (np.float64, np.float32) or not a.flags['C_CONTIGUOUS']:
                        a = np.ascontiguousarray(a, dtype=np.float64)
                    a = torch.from_numpy(a)
                if a.dtype not in (torch.float64, torch.float32):
                    a = a.to(torch.float64)
                # float32 arrays cross the link as float32 (see lossless_float32).  The destination is the ring slot's
                # buffer: the slot is free, `run` has waited for the compute stage of its previous occupant
                buf = bufs[k]
                t = (buf.view(torch.float32)[:a.numel()] if a.dtype == torch.float32 else buf).view(a.shape)
                t.copy_(a, non_blocking=True)
                staged[k] = t
                self.h2d_bytes += t.numel() * t.element_size()
            ev = torch.cuda.Event(enable_timing=self.timeline is not None)
            ev.record(self.h2d)
            if self.timeline is not None:
                self.timeline.append({'h2d': (e0, ev)})
        return staged, ev

    def _to_fields(self, staged):
        """cell-major staging tensors -> month-major Fields (compute stream).  Outside PM, ABCD's tmin is read with NaN
        as 0 (DataLoader loads TempMinFile with nan_to_num; idempotent on an array it cleaned already), while HS reads
        hs_tmin - possibly the same upload - as it is."""
        fields = {}
        for k, t in staged.items():
            f = C.Field.empty(self.s.ncell, self.s.nmonths, self.s.ld)
            fn = C.lib().xan_to_month_major_f32 if t.dtype == self._torch.float32 else C.lib().xan_to_month_major
            nan_to_num = int(k == 'tmin' and self.s.pet != 'pm')
            C.check(fn(C.ptr(t), C.ptr(f.t), self.s.ncell, self.s.nmonths, f.ld, nan_to_num, C.stream_ptr()))
            fields[k] = f
        return fields

    def _mark(self, stream):
        if self.timeline is None:
            return None
        e = self._torch.cuda.Event(enable_timing=True)
        e.record(stream)
        return e

    def _pet(self, fields):
        """The member's PET Field from its month-major forcing (current stream)."""
        s = self.s
        if s.pet == 'pm':
            return pm_mod.run_pmpet_device(s.data_ns(fields), s.ncell, s.nlcs, s.start_yr, s.end_yr, s.water_idx,
                                           s.snow_idx, s.lc_years)
        if s.pet == 'hs':
            return hs_mod.execute_device(fields['hs_tas'], fields['hs_tmax'], fields['hs_tmin'], s.d_lat, s.start_yr)
        if s.pet == 'thornthwaite':
            return th_mod.execute_device(fields['tair'], s.d_lat, s.start_yr)
        return fields['pet']

    def _want(self):
        """The ABCD outputs the back stage and the downloads read: q always, aet / sav when asked for or scanned."""
        dvar = self._drought.var if self._drought is not None else None
        return tuple(k for k, v in (('aet', 'aet'), ('q', 'q'), ('sav', 'soilmoisture'))
                     if v in self.output_vars or k == 'q' or v == dvar)

    def _front(self, uploads):
        """Front stage, per member: wait for its upload, transposes, PET -> ABCD.  `uploads`: [(staged tensors, upload event)].
        Runs on the front stream (beside the routing launch of the group before); returns (PET Fields, ABCD results, event)."""
        s, torch = self.s, self._torch
        compute = torch.cuda.current_stream()
        stream = self.front if self.front is not None else compute
        want = self._want()
        pets, ress = [], []
        with torch.cuda.stream(stream):
            while uploads:
                staged, ev = uploads.pop(0)
                stream.wait_event(ev)     # the first member's PET and runoff run under the second member's upload
                fields = self._to_fields(staged)
                del staged
                pet = self._pet(fields)
                res = abcd_mod.run_device(s.plan, s.d_pars, pet, fields['precip'], fields['tmin'], s.nmonths,
                                          s.runoff_spinup, want=want)
                if stream is not compute:     # allocated on the front stream, read by the routing / output stage
                    for f in [pet] + list(res.values()):
                        f.t.record_stream(compute)
                pets.append(pet)
                ress.append(res)
            ev = torch.cuda.Event()
            ev.record(stream)
        return pets, ress, ev

    def _shared_forcing(self, forcing):
        """The forcing of a parameter ensemble, uploaded, transposed and run through PET once (compute stream): (PET
        Field, month-major forcing Fields)."""
        staged, ev = self._upload(forcing, 0)
        self._torch.cuda.current_stream().wait_event(ev)
        fields = self._to_fields(staged)
        return self._pet(fields), fields

    def _front_sets(self, shared, pars):
        """Front stage of a group of parameter sets (compute stream): ABCD of every table of `pars` [g, n_rows, 5] over
        the shared forcing, one run_device_sets call; returns (PET Fields, ABCD results, event) like `_front`."""
        s, (pet, fields) = self.s, shared
        ress = abcd_mod.run_device_sets(s.plan, pars, pet, fields['precip'], fields['tmin'], s.nmonths, s.runoff_spinup,
                                        want=self._want())
        ev = self._torch.cuda.Event()
        ev.record(self._torch.cuda.current_stream())
        return [pet] * len(ress), ress, ev

    def _back(self, pets, ress):
        """One routing call for the group (with routing) and the basin aggregates per member (compute stream)."""
        s = self.s
        want_chs = 'chstorage' in self.output_vars
        if not s.routing:
            routed = [(None, None, None)] * len(ress)
        elif len(ress) == 1:
            routed = [mrtm_mod.route_device(s.um, ress[0]['q'], s.d_L, s.d_V, s.d_area, s.ndays, s.dt, s.routing_spinup,
                                            want_chs=want_chs)]
        else:
            routed = mrtm_mod.route_device_batch(s.um, [r['q'] for r in ress], s.d_L, s.d_V, s.d_area, s.ndays, s.dt,
                                                 s.routing_spinup, want_chs=want_chs)
        results = []
        for pet, res, (chs, avg, _) in zip(pets, ress, routed):
            out = {'pet': pet, 'aet': res.get('aet'), 'q': res['q'], 'soilmoisture': res.get('sav'), 'chstorage': chs,
                   'avgchflow': avg}
            agg = None
            if self.aggregates:   # basin runoff in km3 / month and basin sum of the mean streamflow, [2, nmonths, n_basins]
                agg = self._torch.empty((self.n_agg_rows, s.nmonths, s.n_basins), dtype=self._torch.float64,
                                        device='cuda')
                C.check(C.lib().xan_basin_sum(s.plan._plan, C.ptr(res['q'].t), C.ptr(s.d_area_km3), s.nmonths,
                                              res['q'].ld, C.ptr(agg[0]), C.stream_ptr()))
                if s.routing:     # without routing [1, nmonths, n_basins]: the runoff row only
                    C.check(C.lib().xan_basin_sum(s.plan._plan, C.ptr(avg.t), None, s.nmonths, avg.ld, C.ptr(agg[1]),
                                                  C.stream_ptr()))
            results.append((out, agg))
        return results

    def _drought_scan(self, out):
        """The member's drought scan (compute stream) on its monthly mm field: its thresholds when the spec has none,
        one xan_drought_scan that adds it to the counts and writes its summary (and its severity / intensity / duration
        grids with spec.fields).  Returns the device tensors to copy back: {'summary': [4, ld], 'thresholds'?:
        [nper, ncell], 'severity'? ...: cell-major [ncell, nmonths]}."""
        from .drought.drought_stats import drought_scan_device, getthresh_device
        d, s, torch = self._drought, self.s, self._torch
        f = out[d.var]
        if f.ld != s.ld:
            raise RuntimeError("ensemble drought: field pitch {} differs from {}".format(f.ld, s.ld))
        res = {'summary': torch.empty((len(DROUGHT_SUMMARY), s.ld), dtype=torch.float64, device='cuda')}
        th = self._drought_th
        if th is None:
            first, end = d.reference_months(s.start_yr, s.end_yr)
            th = res['thresholds'] = getthresh_device(f.t[first:end], s.ncell, d.nper)
        sid = [C.Field.empty(s.ncell, s.nmonths, s.ld) for _ in DROUGHT_FIELDS] if d.fields else None
        drought_scan_device(f.t, s.ncell, th, None if sid is None else [x.t for x in sid], self._drought_count,
                            res['summary'])
        self.n_drought += 1
        for k, x in zip(DROUGHT_FIELDS, sid or ()):
            res[k] = x.to_device_cell_major()
        return res

    def _reduce(self, out):
        """The member's outputs as the spec asks for them (compute stream): yearly aggregation, km3, group sums of q,
        the member added to the across-member statistics and its drought scan.  Returns ({var: Field [ntime][ld]},
        {scale: [ng, ntime]}, drought tensors or None)."""
        s, spec, lib = self.s, self.spec, C.lib()
        drought = self._drought_scan(out) if self._drought is not None else None
        red = {}
        for v in self._reduce_vars:
            f = out[v]
            if spec.output_in_year:
                y = C.Field.empty(s.ncell, self.ntime, f.ld)
                C.check(lib.xan_agg_to_year(C.ptr(f.t), C.ptr(y.t), s.ncell, s.nmonths, f.ld, int(v == 'avgchflow'),
                                            C.stream_ptr()))
                f = y
            if spec.output_unit == 'km3' and v != 'avgchflow':
                dst = f if spec.output_in_year else C.Field.empty(s.ncell, self.ntime, f.ld)   # monthly: keep the original
                C.check(lib.xan_scale_cells(C.ptr(f.t), C.ptr(s.km3_scale()), s.ncell, self.ntime, f.ld, C.ptr(dst.t),
                                            C.stream_ptr()))
                f = dst
            red[v] = f
        groups = {}
        for g, (d_order, d_off, ng) in self._groups.items():
            t = self._torch.empty((ng, self.ntime), dtype=self._torch.float64, device='cuda')
            C.check(lib.xan_group_sum(C.ptr(red['q'].t), C.ptr(d_order), C.ptr(d_off), ng, self.ntime, red['q'].ld,
                                      C.ptr(t), C.stream_ptr()))
            groups[g] = t
        if spec.stats:          # members arrive in order: the sequential sum is numpy's over the stacked members
            self.n_stats += 1
            for v in self.output_vars:
                sm, mm = self._stats_state[v]
                if red[v].ld != s.ld:
                    raise RuntimeError("ensemble statistics: field pitch {} differs from {}".format(red[v].ld, s.ld))
                C.check(lib.xan_ens_stats_update(C.ptr(red[v].t), C.ptr(sm), C.ptr(mm), s.ncell, self.ntime,
                                                 red[v].ld, self.n_stats, C.stream_ptr()))
        if spec.quantiles:      # the member's slot of the stack, device to device on the compute stream
            for v in self.output_vars:
                if red[v].ld != s.ld:
                    raise RuntimeError("ensemble quantiles: field pitch {} differs from {}".format(red[v].ld, s.ld))
                self._stack[v][self.n_stacked].copy_(red[v].t[:self.ntime], non_blocking=True)
            self.n_stacked += 1
        if not spec.member_fields:
            return {}, groups, drought
        return {v: red[v] for v in self.output_vars}, groups, drought

    def _download(self, out, agg):
        torch = self._torch
        compute = torch.cuda.current_stream()
        if self.spec is None:
            fields, groups, drought = {v: out[v] for v in self.output_vars}, {}, None
        else:
            fields, groups, drought = self._reduce(out)
        staged = {v: f.to_device_cell_major() for v, f in fields.items()}      # transposes run on the compute stream
        ev = torch.cuda.Event()
        ev.record(compute)
        self.d2h.wait_event(ev)
        host = {}
        with torch.cuda.stream(self.d2h):
            for v, dev in staged.items():
                dev.record_stream(self.d2h)
                h = C.host_pool.acquire((self.s.ncell, self.ntime))
                h.copy_(dev, non_blocking=True)
                host[v] = h
                self.d2h_bytes += h.numel() * 8
            if agg is not None:
                agg.record_stream(self.d2h)
                h = torch.empty(tuple(agg.shape), dtype=torch.float64, pin_memory=True)
                h.copy_(agg, non_blocking=True)
                host['basin_aggregates'] = h
                self.d2h_bytes += h.numel() * 8
            if groups:
                host['group_sums'] = {}
                for g, t in groups.items():
                    t.record_stream(self.d2h)
                    h = torch.empty(tuple(t.shape), dtype=torch.float64, pin_memory=True)
                    h.copy_(t, non_blocking=True)
                    host['group_sums'][g] = h
                    self.d2h_bytes += h.numel() * 8
            if drought is not None:     # summary and thresholds to pinned tensors, the grids through host_pool
                host['drought'] = {}
                for k, t in drought.items():
                    t.record_stream(self.d2h)
                    h = (C.host_pool.acquire(tuple(t.shape)) if k in DROUGHT_FIELDS
                         else torch.empty(tuple(t.shape), dtype=torch.float64, pin_memory=True))
                    h.copy_(t, non_blocking=True)
                    host['drought'][k] = h[:, :self.s.ncell] if k == 'summary' else h
                    self.d2h_bytes += h.numel() * 8
            done = torch.cuda.Event(enable_timing=self.timeline is not None)
            done.record(self.d2h)
        return host, done

    # ---- across-member statistics -----------------------------------------------------------------------------------
    def stats_partial(self):
        """This runner's accumulators as a flat list [(sum, m2) of var 0, (min, max) of var 0, ...] (None before any
        member): what `merge_stats` combines and `finalize_stats` turns into the statistics."""
        if self._stats_state is None or self.n_stats == 0:
            return None
        return [t for v in self.output_vars for t in self._stats_state[v]]

    def merge_stats(self, a, na, b, nb):
        """Partial `a` of na members absorbs partial `b` of nb members (xan_ens_stats_merge, in place); returns a."""
        for v in range(len(self.output_vars)):
            C.check(C.lib().xan_ens_stats_merge(C.ptr(a[2 * v]), C.ptr(a[2 * v + 1]), C.ptr(b[2 * v]),
                                                C.ptr(b[2 * v + 1]), self.s.ncell, self.ntime, self.s.ld, int(na),
                                                int(nb), C.stream_ptr()))
        return a

    def finalize_stats(self, partial, n):
        """{var: {stat: host ndarray [ncell, ntime]}} of the requested statistics over n members."""
        torch, s, out = self._torch, self.s, {}
        for k, v in enumerate(self.output_vars):
            dev = {st: torch.empty((s.ncell, self.ntime), dtype=torch.float64, device='cuda') for st in self.spec.stats}
            C.check(C.lib().xan_ens_stats_finalize(C.ptr(partial[2 * k]), C.ptr(partial[2 * k + 1]), s.ncell,
                                                   self.ntime, s.ld, int(n), self.spec.ddof,
                                                   *[C.ptr(dev.get(st)) for st in STATS], C.stream_ptr()))
            out[v] = {st: t.cpu().numpy() for st, t in dev.items()}
            self.d2h_bytes += sum(t.numel() * 8 for t in dev.values())
        return out

    # ---- across-member quantiles ------------------------------------------------------------------------------------
    def _alloc_stack(self, n):
        """The member stack [n, ntime, ld] of every output variable, 8 B per cell, time step, variable and member: made
        before the pipeline starts (and reused by a later run of as many members), refused if it cannot fit."""
        torch, s = self._torch, self.s
        if n > C.ENS_MAX_MEMBERS:
            raise C.ValidationException("quantiles over {} members (at most {})".format(n, C.ENS_MAX_MEMBERS))
        shape = (n, self.ntime, s.ld)
        if self._stack is not None and tuple(self._stack[self.output_vars[0]].shape) == shape:
            return
        self._stack = None
        need = 8 * n * self.ntime * s.ld * len(self.output_vars)
        # free to the driver plus what torch's caching allocator holds unused
        free = torch.cuda.mem_get_info()[0] + torch.cuda.memory_reserved() - torch.cuda.memory_allocated()
        if need > free:
            raise C.ValidationException(
                "the member stack of the quantiles needs {:,} bytes ({} members x {} time steps x {} cells (pitch {}) x "
                "{} variables x 8 B), the device has {:,} free".format(need, n, self.ntime, s.ncell, s.ld,
                                                                       len(self.output_vars), free))
        self._stack = {v: torch.empty(shape, dtype=torch.float64, device='cuda') for v in self.output_vars}

    def member_stack(self):
        """{var: device tensor [n, ntime, ld]}: the reduced fields of the members of the last `run`, in member order
        (None without quantiles or before any member) - what `finalize_quantiles` takes."""
        if self._stack is None or self.n_stacked == 0:
            return None
        return {v: t[:self.n_stacked] for v, t in self._stack.items()}

    def _chunk_steps(self, n):
        return max(1, min(self.ntime, QUANTILE_CHUNK_BYTES // (8 * n * self.s.ld * len(self.output_vars))))

    def _assembled(self, n, fill):
        """Generator of (t0, {var: [n, nt, ld]}) over the time steps in chunks that keep the buffers within
        QUANTILE_CHUNK_BYTES (at least one step); fill(var, t0, t1, buf) writes the members' rows of a chunk."""
        torch, ld = self._torch, self.s.ld
        chunk = self._chunk_steps(n)
        bufs = {v: torch.empty(n * chunk * ld, dtype=torch.float64, device='cuda') for v in self.output_vars}
        for t0 in range(0, self.ntime, chunk):
            t1 = min(self.ntime, t0 + chunk)
            views = {v: b[:n * (t1 - t0) * ld].view(n, t1 - t0, ld) for v, b in bufs.items()}
            for v, buf in views.items():
                fill(v, t0, t1, buf)
            yield t0, views

    def _quantiles(self, n, blocks):
        """blocks: (t0, {var: member stack of the steps from t0}) covering all steps -> finalize_quantiles' result."""
        torch, s, levels = self._torch, self.s, self.spec.quantiles
        if not 1 <= n <= C.ENS_MAX_MEMBERS:
            raise C.ValidationException("quantiles over {} members (1 to {})".format(n, C.ENS_MAX_MEMBERS))
        dev = {v: torch.empty((len(levels), s.ncell, self.ntime), dtype=torch.float64, device='cuda')
               for v in self.output_vars}
        for t0, blk in blocks:
            for v in self.output_vars:
                member_quantiles(blk[v], s.ncell, levels, dev[v], t0)
        out = {'levels': levels, 'n_members': n}
        for v, t in dev.items():
            out[v] = t.cpu().numpy()
            self.d2h_bytes += t.numel() * 8
        return out

    def finalize_quantiles(self, stacks):
        """{'levels': spec.quantiles, 'n_members': N, var: host ndarray [nq, ncell, ntime]}: numpy.quantile over the
        members of the `member_stack()`s of one or several runners, given in member order.  One stack is read where it
        lies; several are brought together a chunk of time steps at a time by device-to-device copies."""
        stacks = [st for st in stacks if st is not None]
        counts = [int(st[self.output_vars[0]].shape[0]) for st in stacks]
        if len(stacks) == 1:
            return self._quantiles(counts[0], [(0, stacks[0])])

        def fill(v, t0, t1, buf):
            o = 0
            for st, k in zip(stacks, counts):
                buf[o:o + k].copy_(st[v][:, t0:t1])
                o += k
        return self._quantiles(sum(counts), self._assembled(sum(counts), fill))

    def gather_quantiles(self, counts):
        """Under torch.distributed (counts[r] members on rank r, contiguous blocks in rank order): rank 0 gathers the
        member stacks of all ranks one chunk of time steps at a time (sharding.gather_rows_to_rank0) and returns what
        `finalize_quantiles` returns for all members; the other ranks send their rows and return None."""
        import torch.distributed as dist
        n, mine = sum(counts), self.member_stack()

        def local(v, t0, t1):
            return None if mine is None else mine[v][:, t0:t1]
        if dist.get_rank() != 0:
            chunk = self._chunk_steps(n)
            for t0 in range(0, self.ntime, chunk):
                for v in self.output_vars:
                    sharding.gather_rows_to_rank0(local(v, t0, t0 + chunk), counts)
            return None
        return self._quantiles(n, self._assembled(
            n, lambda v, t0, t1, buf: sharding.gather_rows_to_rank0(local(v, t0, t1), counts, buf)))

    # ---- across-member drought frequency ----------------------------------------------------------------------------
    def drought_partial(self):
        """[int32 device tensor [nmonths, ld]]: members of the last `run` in drought per month and cell (None without
        drought or before any member) - what `merge_drought_counts` combines and `finalize_drought` reports."""
        if self._drought_count is None or self.n_drought == 0:
            return None
        return [self._drought_count]

    def finalize_drought(self, partial, n):
        """{'members_in_drought': int32 [ncell, nmonths], 'frequency': members_in_drought / n, 'n_members': n}."""
        cnt = partial[0][:, :self.s.ncell].t().contiguous().cpu().numpy()
        self.d2h_bytes += cnt.nbytes
        return {'members_in_drought': cnt, 'frequency': cnt / n, 'n_members': int(n)}

    # ---- driver ----------------------------------------------------------------------------------------------------------
    def run(self, members, parameter_sets=None):
        """Generator: yields (index, {variable: host ndarray [ncell, nmonths], 'basin_aggregates': [n_agg_rows, nmonths,
        n_basins]}) in member order; the next members are being uploaded and a group of `group` members computed while
        the outputs of the group before are handed out.  With a spec the grids are [ncell, ntime] (none without member_fields), the
        result has 'group_sums': {scale: [ngroups, ntime]}, and each member is added to the across-member statistics
        (`stats_partial` / `finalize_stats` once the generator is exhausted), its reduced fields kept on the device for
        the quantiles (`member_stack` / `finalize_quantiles`), and with spec.drought the result has 'drought':
        {'summary': {name: [ncell]}, 'thresholds'?: [nper, ncell], 'severity' / 'intensity' / 'duration'?:
        [ncell, nmonths]} and the member is added to the drought counts (`drought_partial` / `finalize_drought`).

        With `parameter_sets` (float64 [P, n_rows, 5], see `parameter_sets`) `members` is ONE forcing dict, uploaded,
        transposed and run through PET once before the loop, and item k is ABCD parameter table k over it: a group's
        front stage is one run_device_sets call for its tables (pairs with routing, PARAMETER_SETS_PER_LAUNCH without)."""
        torch = self._torch
        shared = None
        if parameter_sets is None:
            members = list(members)
            n, g = len(members), self.group
        else:
            n, g = len(parameter_sets), (self.group if self.s.routing else PARAMETER_SETS_PER_LAUNCH)
        if not n:
            return
        compute = torch.cuda.current_stream()
        depth = self.prefetch_depth
        # pinned output buffers in flight: the group being computed, the group before it on its way to the host, and the
        # results the caller still holds from the last hand-out - allocated before the pipeline starts, not inside it
        in_flight, grids = min(3 * g, n + g), {}          # cells x time steps -> pinned grids the pipeline holds
        if self.spec is None or self.spec.member_fields:
            grids[self.ntime] = in_flight * len(self.output_vars)
        if self._drought is not None and self._drought.fields:
            grids[self.s.nmonths] = grids.get(self.s.nmonths, 0) + in_flight * len(DROUGHT_FIELDS)
        for nt, count in grids.items():
            C.host_pool.reserve((self.s.ncell, nt), count)
        self.n_stats = self.n_stacked = self.n_drought = 0
        if self._drought is not None:      # 4 B per month and cell, made before the pipeline starts
            if self._drought_count is None:
                self._drought_count = torch.zeros((self.s.nmonths, self.s.ld), dtype=torch.int32, device='cuda')
            else:
                self._drought_count.zero_()
        if self.spec is not None and self.spec.quantiles:
            self._alloc_stack(n)
        if self.spec is not None and self.spec.stats and self._stats_state is None:
            self._stats_state = {v: tuple(torch.empty((self.ntime, self.s.ld, 2), dtype=torch.float64, device='cuda')
                                          for _ in range(2)) for v in self.output_vars}
        if parameter_sets is not None:
            shared = self._shared_forcing(members)
            d_sets = torch.from_numpy(np.ascontiguousarray(parameter_sets, dtype=np.float64)).cuda()
            if self.timeline is not None:      # every set's entry starts at the one upload
                self.timeline.extend(dict(self.timeline[-1]) for _ in range(n - 1))
        uploaded, next_up = {}, 0
        pending = []              # (index, host tensors, done event) of the members whose outputs are in flight
        computed = {}             # member -> completion event of its group's compute stage, to bound the uploads' run-ahead

        def pump(k):              # uploads of the members up to k + depth; member j waits for the compute of member j - depth - g
            nonlocal next_up
            while shared is None and next_up < n and next_up <= k + depth:
                old = next_up - depth - g
                if old >= 0:
                    computed[old].synchronize()
                uploaded[next_up] = self._upload(members[next_up], next_up % (depth + g))
                next_up += 1
        fronts = {}

        def start_front(k0):      # front stage of the group starting at member k0
            ks = list(range(k0, min(n, k0 + g)))
            if shared is not None:
                fronts[k0] = self._front_sets(shared, d_sets[k0:ks[-1] + 1])
                return
            if ks[-1] not in uploaded:
                pump(ks[-1] - depth)
            fronts[k0] = self._front([uploaded.pop(k) for k in ks])
        pump(g - 1)
        start_front(0)
        for k0 in range(0, n, g):
            ks = list(range(k0, min(n, k0 + g)))
            pets, ress, fev = fronts.pop(k0)
            c0 = self._mark(compute)
            compute.wait_event(fev)
            results = self._back(pets, ress)
            del pets, ress
            if k0 + g < n:        # enqueued behind this group's routing launch, runs beside it on the device
                start_front(k0 + g)
            downloads = [self._download(out, agg) for out, agg in results]
            del results
            cev = torch.cuda.Event(enable_timing=self.timeline is not None)
            cev.record(compute)
            for k, (host, done) in zip(ks, downloads):
                computed[k] = cev
                if self.timeline is not None:
                    self.timeline[k]['compute'] = (c0, cev)
                    self.timeline[k]['done'] = done
            pump(ks[-1])
            for p in pending:
                yield self._finish(p)
            pending = [(k, host, done) for k, (host, done) in zip(ks, downloads)]
        for p in pending:
            yield self._finish(p)

    @staticmethod
    def _finish(p):
        k, host, done = p
        done.synchronize()
        res = {}
        for v, h in host.items():
            if v == 'group_sums':
                res[v] = {g: t.numpy() for g, t in h.items()}
            elif v == 'drought':
                res[v] = {k: (dict(zip(DROUGHT_SUMMARY, t.numpy())) if k == 'summary'
                              else C.host_pool.as_array(t) if k in DROUGHT_FIELDS else t.numpy()) for k, t in h.items()}
            else:
                res[v] = C.host_pool.as_array(h) if v != 'basin_aggregates' else h.numpy()
        return k, res


def run_ensemble(statics, members, output_vars=('q', 'avgchflow'), aggregates=True, on_result=None, spec=None):
    """
    Run every member (this rank's share when torch.distributed is initialised: a contiguous block per rank,
    sharding.partition_members).
    Returns {member index: result dict}; with `on_result(index, result)` given the results are handed to it instead of
    being kept (a 64-member ensemble of 1,032 months is 2 x 36 GB of output).  On every rank the returned dict also has
    the key 'basin_aggregates': [n_members, 2, nmonths, n_basins] of ALL members (all-gather over NCCL); without
    routing (EnsembleStatics(routing=False)) it is [n_members, 1, nmonths, n_basins], the basin runoff in km3 / month.

    `spec` (OutputSpec) reduces the outputs on the device before they are copied back; without it every member's
    monthly grids come back as they are.  With it:
      * a member's result holds the grids {var: [ncell, ntime]} (ntime = nyears with yearly output) only if
        spec.member_fields, and 'group_sums': {scale: [ngroups, ntime]};
      * the returned dict has 'group_sums': {scale: [n_members, ngroups, ntime]} of all members on every rank, and on
        rank 0 'ensemble_stats': {var: {stat: [ncell, ntime]}, 'n_members': N}.
    The statistics are accumulated on the device member by member (fp64 accumulators of 32 B per cell and time step
    and variable: 2.2 GB per monthly variable at 67,420 cells x 1,032 months); each rank keeps the partial of its
    members and rank 0 merges them in rank order (Chan et al.).  The result is deterministic for a given number of
    ranks; min / max do not depend on it, mean and std may differ in the last bits between rank counts.

    With spec.quantiles rank 0 also gets 'ensemble_quantiles': {'levels': spec.quantiles, 'n_members': N,
    var: [nq, ncell, ntime]}, numpy.quantile(members, levels, axis=0) bitwise.  Every member's reduced field stays on
    the device (8 B per cell, time step, variable and member: 2.97 GB per yearly variable of 64 members x 86 years,
    35.6 GB per monthly variable of 64 members x 1,032 months, at 67,420 cells), checked against the free memory
    before the run; at most 256 members.  Rank 0 gathers the members of all ranks point to point in rank order, a
    chunk of time steps at a time, and selects over them: the quantiles do not depend on the member order, so they
    are bitwise the same for every number of ranks.

    With spec.drought every member's result has 'drought' (see EnsembleRunner.run), the returned dict has
    'drought_summary': [n_members, 4, ncell] (DROUGHT_SUMMARY: drought months, events, longest duration, peak severity)
    of all members in member order on every rank, and rank 0 gets 'ensemble_drought': {'members_in_drought': int32
    [ncell, nmonths], 'frequency': members_in_drought / N, 'n_members': N}.  Each rank counts its members on the device
    (int32 [nmonths, ld], 278 MB at 67,420 cells x 1,032 months) and rank 0 adds the counts of the other ranks: integer
    sums are exact, so the counts and the frequency are bitwise the same for every number of ranks.
    """
    members = list(members)
    return _run_sharded(statics, len(members), lambda runner, mine: runner.run([members[i] for i in mine]),
                        output_vars, aggregates, on_result, spec)


def run_parameter_ensemble(statics, forcing, parameter_sets, output_vars=('q', 'avgchflow'), aggregates=True,
                           on_result=None, spec=None):
    """
    A parameter ensemble: ABCD parameter table k (perturbations of a calibrated table, samples of a GLUE-style search)
    over ONE forcing is "member k" of `run_ensemble`, and the return value has exactly its shape - per-set results,
    'basin_aggregates' [P, rows, nmonths, n_basins], 'group_sums', 'ensemble_stats', 'ensemble_quantiles',
    'drought_summary', 'ensemble_drought' and 'stats' (h2d_bytes, d2h_bytes, members_local).

      forcing         one member dict with the keys of forcing_fields(statics.pet); it crosses the host -> device link
                      and goes through PET once (once per rank under torch.distributed)
      parameter_sets  one [P, n_rows, 4 or 5] array or a sequence of [n_rows, 4 or 5] tables (see `parameter_sets`);
                      statics.abcd_pars is not run: it only fixes n_rows, the row count every table must have

    Set k is bit-identical to the plug-in calls on table k (PET -> abcd_execute(..., pars_k, ...) -> mrtm.route) and
    does not depend on the other sets.  ABCD runs several tables per launch (xan_abcd_run_sets); routing, the output
    options and the across-set reductions are those of `run_ensemble`, and under torch.distributed the sets are dealt
    to the ranks as members are.  'pet' is not an output: it is the same for every set.
    """
    if 'pet' in output_vars:
        raise C.ValidationException("'pet' is not an output of a parameter ensemble: PET comes from the one forcing and "
                                    "is the same for every parameter set (run_ensemble with the forcing returns it)")
    missing = [k for k in forcing_fields(statics.pet) if k not in forcing]
    if missing:
        raise C.ValidationException("the forcing lacks {} (pet={!r})".format(missing, statics.pet))
    sets = _parameter_sets(parameter_sets, statics.d_pars.shape[0])
    return _run_sharded(statics, len(sets), lambda runner, mine: runner.run(forcing, parameter_sets=sets[mine]),
                        output_vars, aggregates, on_result, spec)


def _run_sharded(statics, n_members, run_local, output_vars, aggregates, on_result, spec):
    """run_ensemble's driver over n_members items, this rank's share run by run_local(runner, indices)."""
    torch = C.torch_cuda()
    import torch.distributed as dist
    if spec is not None and spec.quantiles and n_members > C.ENS_MAX_MEMBERS:
        raise C.ValidationException("quantiles over {} members (at most {})".format(n_members, C.ENS_MAX_MEMBERS))
    dist_on = dist.is_available() and dist.is_initialized()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist_on else (0, 1)
    parts = sharding.partition_members(n_members, world)
    mine = [int(i) for i in parts[rank]]
    runner = EnsembleRunner(statics, output_vars, aggregates, spec=spec)
    results = {}
    agg_local = torch.zeros((len(mine), runner.n_agg_rows, statics.nmonths, statics.n_basins), dtype=torch.float64)
    groups = spec.group_sums if spec is not None else ()
    grp_local = {g: torch.zeros((len(mine), statics.group_table(g)[2], runner.ntime), dtype=torch.float64)
                 for g in groups}
    drought = spec is not None and spec.drought is not None
    dr_local = torch.zeros((len(mine), len(DROUGHT_SUMMARY), statics.ncell), dtype=torch.float64) if drought else None
    for j, res in run_local(runner, mine):
        if aggregates:
            agg_local[j] = torch.from_numpy(res['basin_aggregates'])
        for g in groups:
            grp_local[g][j] = torch.from_numpy(res['group_sums'][g])
        if drought:
            dr_local[j] = torch.from_numpy(np.stack([res['drought']['summary'][k] for k in DROUGHT_SUMMARY]))
        if on_result is not None:
            on_result(mine[j], res)
        else:
            results[mine[j]] = res
    if aggregates:      # every rank gets the basin aggregates of all members
        results['basin_aggregates'] = sharding.gather_ragged_rows(mine, agg_local.cuda(), n_members).cpu().numpy()
    if groups:
        results['group_sums'] = {g: sharding.gather_ragged_rows(mine, grp_local[g].cuda(), n_members).cpu().numpy()
                                 for g in groups}
    if drought:
        results['drought_summary'] = sharding.gather_ragged_rows(mine, dr_local.cuda(), n_members).cpu().numpy()
    if drought and n_members:
        partial = sharding.fold_to_rank0(runner.drought_partial(), [len(p) for p in parts], merge_drought_counts)
        if rank == 0:
            results['ensemble_drought'] = runner.finalize_drought(partial, n_members)
    if spec is not None and spec.stats and n_members:
        partial = sharding.fold_to_rank0(runner.stats_partial(), [len(p) for p in parts], runner.merge_stats)
        if rank == 0:
            results['ensemble_stats'] = runner.finalize_stats(partial, n_members)
            results['ensemble_stats']['n_members'] = n_members
    if spec is not None and spec.quantiles and n_members:
        if world > 1:
            quant = runner.gather_quantiles([len(p) for p in parts])
        else:
            quant = runner.finalize_quantiles([runner.member_stack()])
        if rank == 0:
            results['ensemble_quantiles'] = quant
    results['stats'] = {'h2d_bytes': runner.h2d_bytes, 'd2h_bytes': runner.d2h_bytes, 'members_local': len(mine)}
    if runner.timeline:      # ms relative to the first upload: (h2d start, end), (compute start, end), outputs on the host
        torch.cuda.synchronize()
        t0 = runner.timeline[0]['h2d'][0]
        results['stats']['timeline'] = [
            {'h2d': [round(t0.elapsed_time(e), 1) for e in m['h2d']],
             'compute': [round(t0.elapsed_time(e), 1) for e in m['compute']],
             'done': round(t0.elapsed_time(m['done']), 1)} for m in runner.timeline if 'compute' in m]
    return results
