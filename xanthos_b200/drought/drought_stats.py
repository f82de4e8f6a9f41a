"""
Drought statistics on the device-resident fields - counterpart of xanthos/drought/drought_stats.py.

Same class, method names, argument meaning, outputs and files as the reference (`DroughtStats(settings, runoff,
soil_moisture)`, `calculate_thresholds`, `droughtstats`, `getthresh`).  The reference transposes its [ncell, nmonths]
arrays to [ntime, ngrid] first (drought_stats.py:37-44); that IS the month-major layout of this library, so an
array a CUDA stage returned is used where it lies in HBM, and a host [ntime, ngrid] array is uploaded as it is.
Kernels: xan_drought_stats (one thread per cell walks the months), xan_drought_thresholds (numpy.percentile,
method 'linear', per (period, cell)) - both bit-identical to numpy.  There is no CPU fallback.
"""

import logging
import os

import numpy as np

from .. import _cuda as C

MONTHS_IN_YEAR = 12


def _as_time_major(x):
    """[ntime, ngrid] host array / cuda tensor / Field -> (tensor [ntime, ld], ngrid)."""
    torch = C.torch_cuda()
    if isinstance(x, C.Field):
        return x.t, x.ncell
    if isinstance(x, torch.Tensor):
        return x.to(device='cuda', dtype=torch.float64).contiguous(), int(x.shape[1])
    a = np.ascontiguousarray(x, dtype=np.float64)
    return torch.from_numpy(a).to('cuda', non_blocking=True), a.shape[1]


def virtual_index(n, q):
    """numpy's position of the q-quantile among n sorted samples for method 'linear': (n - 1) q -> (floor, fraction)."""
    vi = (n - 1) * q
    prev = int(np.floor(vi))
    return prev, float(vi - prev)


def getthresh_device(hist, ngrid, nper, quantile=0.1):
    """hist: cuda tensor [ntime, ld] -> cuda tensor [nper, ngrid]."""
    torch = C.torch_cuda()
    ntime, ld = int(hist.shape[0]), int(hist.shape[1])
    nyear = int(ntime / nper)
    if nyear < 1 or nyear * nper != ntime:
        raise ValueError("cannot reshape array of size {} into shape ({},{},{})".format(ntime * ngrid, nyear, nper, ngrid))
    q = float(np.true_divide(quantile * 100, 100))     # np.percentile divides the percentage by 100
    prev, gamma = virtual_index(nyear, q)
    out = torch.empty((nper, ngrid), dtype=torch.float64, device='cuda')
    C.check(C.lib().xan_drought_thresholds(C.ptr(hist), ngrid, ntime, ld, nper, prev, gamma, C.ptr(out), ngrid,
                                           C.stream_ptr()))
    return out


def droughtstats_device(hydro, ngrid, thresh):
    """hydro: cuda tensor [ntime, ld]; thresh: cuda tensor [K, ld_t] -> (S, I, D) cuda tensors [ntime, ld]."""
    torch = C.torch_cuda()
    ntime, ld = int(hydro.shape[0]), int(hydro.shape[1])
    if int(thresh.shape[1]) < ngrid:
        raise C.ValidationException("drought thresholds have {} cells, the hydrological output {}".format(
            int(thresh.shape[1]), ngrid))
    S, I, D = (torch.empty((ntime, ld), dtype=torch.float64, device='cuda') for _ in range(3))
    C.check(C.lib().xan_drought_stats(C.ptr(hydro), C.ptr(thresh), ngrid, ntime, ld, int(thresh.shape[0]),
                                      int(thresh.shape[1]), C.ptr(S), C.ptr(I), C.ptr(D), C.stream_ptr()))
    return S, I, D


def drought_scan_device(hydro, ngrid, thresh, sid=None, count=None, summary=None):
    """xan_drought_scan: hydro cuda [ntime, ld], thresh cuda [K, ld_t]; sid = (S, I, D) cuda [ntime, ld] written as
    droughtstats_device writes them; count int32 cuda [ntime, ld] += months in drought and summary cuda [4, ld] = the
    drought months, events, longest duration and peak severity of every cell.  At least one of sid / count."""
    ntime, ld = int(hydro.shape[0]), int(hydro.shape[1])
    if int(thresh.shape[1]) < ngrid or thresh.stride(1) != 1:
        raise C.ValidationException("drought thresholds {} (strides {}) are not rows of at least {} cells".format(
            tuple(thresh.shape), thresh.stride(), ngrid))
    S, I, D = sid if sid is not None else (None, None, None)
    C.check(C.lib().xan_drought_scan(C.ptr(hydro), C.ptr(thresh), ngrid, ntime, ld, int(thresh.shape[0]),
                                     int(thresh.stride(0)), C.ptr(S), C.ptr(I), C.ptr(D), C.ptr(count), C.ptr(summary),
                                     C.stream_ptr()))


class DroughtStats:
    """Analyze drought impacts based on runoff or soil moisture (Sheffield and Wood 2008)."""

    MONTHS_IN_YEAR = MONTHS_IN_YEAR

    def __init__(self, settings, runoff, soil_moisture):
        var = settings.drought_var.lower()
        if var == 'q':
            src = runoff
        elif var == 'soilmoisture':
            src = soil_moisture
        else:
            raise ValueError("Invalid drought variable specified (must be 'q' or 'soilmoisture')")
        # [ncell, nmonths] as Components holds it; its device copy (if a CUDA stage returned it) is month-major already
        field = C.as_field(src)
        output_path = os.path.join(settings.OutputFolder, "drought_{}_{}".format("{}", settings.OutputNameStr))

        if settings.drought_thresholds is None:
            logging.info("\tCalculating drought thresholds")
            thresholds = self.calculate_thresholds(field, settings)
            np.save(output_path.format("thresholds"), thresholds)
        else:
            logging.info("\tCalculating drought statistics")
            threshvals = np.load(settings.drought_thresholds)
            severity, intensity, duration = self.droughtstats(field, threshvals)
            from ..data_writer.out_writer import OutWriter
            out_writer = OutWriter(settings, 0, {})
            for varname, arr in zip(["severity", "intensity", "duration"], [severity, intensity, duration]):
                # the reference writes arr.T with the time index as column name (drought_stats.py:60-63)
                out_writer.write_data(output_path.format(varname), varname, np.ascontiguousarray(arr.T),
                                      col_names=[str(x) for x in range(arr.shape[0])], index_base=0)

    @classmethod
    def calculate_thresholds(cls, histout, settings):
        """histout [ntime x ngrid] -> quantile array [nper x ngrid] (drought_stats.py:67-83; the slice end
        (eyear + 1 - syear) * 12 is an index, not a length, exactly as in the reference)."""
        t, ngrid = _as_time_major(histout)
        syear, eyear = settings.threshold_start_year, settings.threshold_end_year
        smonth = (syear - settings.StartYear) * cls.MONTHS_IN_YEAR
        emonth = (eyear + 1 - syear) * cls.MONTHS_IN_YEAR
        return getthresh_device(t[smonth:emonth], ngrid, settings.threshold_nper).cpu().numpy()

    def droughtstats(self, hydroout, threshvals):
        """(S, I, D) [ntime x ngrid] from hydroout [ntime x ngrid] and threshvals [K x ngrid] (drought_stats.py:85-148)."""
        t, ngrid = _as_time_major(hydroout)
        th, _ = _as_time_major(np.asarray(threshvals, dtype=np.float64))
        S, I, D = droughtstats_device(t, ngrid, th)
        return tuple(x[:, :ngrid].cpu().numpy() for x in (S, I, D))

    @staticmethod
    def getthresh(histout, nper, quantile=0.1):
        """Quantile thresholds [nper x ngrid] of a reference period [ntime x ngrid] (drought_stats.py:150-171)."""
        t, ngrid = _as_time_major(histout)
        return getthresh_device(t, ngrid, nper, quantile).cpu().numpy()
