"""
ctypes binding of libxanthos_b200.so (the C ABI declared in include/xanthos_b200.h) and the
device-buffer plumbing around it.

PyTorch is used for exactly three things: owning device memory (`torch.empty(..., device='cuda')`),
pinned host staging buffers, and CUDA streams.  All arithmetic of the hot path happens inside the
library's hand-written sm_100a kernels.  There is NO CPU fallback: if the shared library or a CUDA
device is missing, every compute call raises.
"""

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libxanthos_b200.so')

XAN_OK, XAN_E_INVALID, XAN_E_CUDA, XAN_E_SPINUP, XAN_E_NOMEM = 0, -1, -2, -3, -4
MRTM_AUTO, MRTM_GRID, MRTM_TREE, MRTM_SKEW = 0, 1, 2, 3
PM_MAX_CLASSES = 32
ENS_MAX_MEMBERS, ENS_MAX_LEVELS = 256, 64      # XAN_ENS_MAX_MEMBERS / XAN_ENS_MAX_LEVELS (xan_ens_quantiles)
DROUGHT_MAX_YEARS = 1024                        # MAX_YEARS of xan_drought_thresholds: samples per (period, cell)
ABCD_MAX_SETS = 8                               # XAN_ABCD_MAX_SETS: parameter tables per xan_abcd_run_sets call


class ValidationException(Exception):
    """Same role as xanthos.data_reader.data_load.ValidationException (data_load.py:24)."""


class LibraryMissing(RuntimeError):
    """libxanthos_b200.so has not been built (python -c 'import __graft_entry__ as g; g.build()')."""


class PmTables(ctypes.Structure):
    _fields_ = [('nlcs', c_int), ('water_idx', c_int), ('snow_idx', c_int)] + \
               [(k, POINTER(c_double)) for k in ('cL', 'beta', 'rslimit', 'Tminopen', 'Tminclose', 'VPDclose',
                                                 'VPDopen', 'RBLmin', 'RBLmax', 'rc', 'emiss',
                                                 'alpha', 'lai', 'laimin', 'laimax')]


# every exported symbol of include/xanthos_b200.h: name -> (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    'xan_version': (c_int, []),
    'xan_last_error': (c_char_p, []),
    'xan_device_info': (c_int, [POINTER(c_int)] * 3),
    'xan_to_month_major': (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    'xan_to_month_major_f32': (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    'xan_to_cell_major': (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    'xan_hs_pet': (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'xan_thornthwaite_pet': (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'xan_thornthwaite_daylight': (c_int, [_P, _P, c_int, _P]),
    'xan_pm_pet': (c_int, [_P] * 9 + [POINTER(PmTables), POINTER(c_int), _P, c_int, c_int, c_int, c_int, _P]),
    'xan_abcd_plan_create': (_P, [POINTER(c_int), c_int, c_int]),
    'xan_abcd_plan_destroy': (None, [_P]),
    'xan_abcd_run': (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    'xan_abcd_run_sets': (c_int, [_P, c_int, c_int, _P, _P, _P, _P, c_int, c_int, c_int, POINTER(_P), POINTER(_P),
                                  POINTER(_P), _P]),
    'xan_abcd_kge_batch': (c_int, [_P, POINTER(c_int), c_int, c_int, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int,
                                   c_int, _P, _P, _P]),
    'xan_mrtm_downstream': (c_int, [POINTER(c_double), POINTER(c_double), c_int, c_int, c_int, POINTER(c_int64)]),
    'xan_mrtm_upstream': (c_int, [POINTER(c_double), POINTER(c_int64), c_int, c_int, c_int, POINTER(c_int64)]),
    'xan_mrtm_plan_create': (_P, [POINTER(c_int64), c_int, c_int, c_int]),
    'xan_mrtm_plan_destroy': (None, [_P]),
    'xan_mrtm_plan_um_nnz': (c_int, [_P]),
    'xan_mrtm_plan_um': (c_int, [_P, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]),
    'xan_mrtm_plan_info': (c_int, [_P, POINTER(c_int)]),
    'xan_mrtm_plan_packing': (c_int, [_P, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    'xan_mrtm_skew_info': (c_int, [_P, POINTER(c_int)]),
    'xan_mrtm_skew_window': (c_int, [_P, c_int, c_int, POINTER(c_int)]),
    'xan_mrtm_skew_tables': (c_int, [_P] + [POINTER(c_int)] * 10),
    'xan_mrtm_route': (c_int, [_P, _P, _P, _P, _P, _P, POINTER(c_int), c_int, c_int, c_int, c_double, c_int,
                               _P, _P, _P, _P]),
    'xan_mrtm_route_batch': (c_int, [_P, c_int, POINTER(_P), _P, _P, _P, POINTER(_P), POINTER(c_int), c_int, c_int,
                                     c_int, c_double, c_int, POINTER(_P), POINTER(_P), POINTER(_P), _P]),
    'xan_hargreaves_pet': (c_int, [_P, _P, _P, POINTER(c_double), POINTER(c_double), POINTER(c_int), _P, c_int, c_int,
                                   c_int, _P]),
    'xan_gwam_run': (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    'xan_agg_to_year': (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    'xan_basin_sum': (c_int, [_P, _P, _P, c_int, c_int, _P, _P]),
    'xan_drought_stats': (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    'xan_drought_scan': (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    'xan_drought_thresholds': (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_double, _P, c_int, _P]),
    'xan_group_sum': (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P]),
    'xan_year_sum_scaled': (c_int, [_P, _P, c_int, c_int, c_int, _P, _P]),
    'xan_scale_cells': (c_int, [_P, _P, c_int, c_int, c_int, _P, _P]),
    'xan_ens_stats_update': (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    'xan_ens_stats_merge': (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    'xan_ens_stats_finalize': (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    'xan_ens_quantiles': (c_int, [_P, ctypes.c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  POINTER(c_int), POINTER(c_double), _P, _P]),
    'xan_de_init': (c_int, [_P, c_int, c_int, c_int, ctypes.c_ulonglong, _P]),
    'xan_de_trial': (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, ctypes.c_ulonglong, c_int, c_double,
                             c_double, c_double, _P, _P, _P]),
    'xan_de_select': (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P, c_double, c_double, c_int, _P, _P]),
}

_lib = None

# kernels launched by each entry point (the claim behind bench.py's "gpu_launches")
KERNELS_PER_CALL = {
    'xan_to_month_major': 1, 'xan_to_month_major_f32': 1, 'xan_to_cell_major': 1, 'xan_hs_pet': 2, 'xan_thornthwaite_pet': 2,
    'xan_thornthwaite_daylight': 1, 'xan_pm_pet': 1, 'xan_abcd_run': 3, 'xan_abcd_run_sets': 3,
    'xan_abcd_kge_batch': 1,
    'xan_mrtm_route': 1, 'xan_mrtm_route_batch': 1, 'xan_hargreaves_pet': 1, 'xan_gwam_run': 1, 'xan_agg_to_year': 1, 'xan_basin_sum': 1,
    'xan_drought_stats': 1, 'xan_drought_scan': 1, 'xan_drought_thresholds': 1, 'xan_group_sum': 1, 'xan_year_sum_scaled': 1,
    'xan_scale_cells': 1, 'xan_ens_stats_update': 1, 'xan_ens_stats_merge': 1, 'xan_ens_stats_finalize': 1,
    'xan_ens_quantiles': 1, 'xan_de_init': 1, 'xan_de_trial': 1, 'xan_de_select': 1,
}
launch_count = 0


class _CountingLib:
    """Thin proxy over the CDLL that counts kernel launches per entry point."""

    def __init__(self, cdll):
        self._cdll = cdll

    def __getattr__(self, name):
        fn = getattr(self._cdll, name)
        n = KERNELS_PER_CALL.get(name, 0)
        if n == 0:
            return fn

        def counted(*args):
            global launch_count
            launch_count += n
            return fn(*args)
        return counted


def lib():
    """The loaded shared library (raises LibraryMissing when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise LibraryMissing("{} not found - build it with `make -C xanthos_b200/csrc` "
                                 "(or __graft_entry__.build()); there is no CPU fallback".format(LIB_PATH))
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = _CountingLib(L)
    return _lib


def check(rc):
    """Map a C-ABI status to the exception type the reference raises for the same condition."""
    if rc == XAN_OK:
        return
    msg = lib().xan_last_error().decode('utf-8', 'replace')
    if rc == XAN_E_SPINUP:
        raise IndexError(msg)                       # abcd.py:253-266
    if rc == XAN_E_INVALID:
        raise ValidationException(msg)
    raise RuntimeError("libxanthos_b200: {} (code {})".format(msg, rc))


def check_ptr(p):
    if not p:
        raise ValidationException(lib().xan_last_error().decode('utf-8', 'replace'))
    return p


# ------------------------------------------------------------------------------------------------
# torch plumbing
# ------------------------------------------------------------------------------------------------
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("xanthos_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch


def device_available():
    """True when a CUDA device is present (used only to choose pinned host buffers for file input)."""
    try:
        import torch
        return bool(torch.cuda.is_available())
    except Exception:
        return False


def stream_ptr():
    torch = torch_cuda()
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def padded_ld(ncell):
    """Row pitch of month-major fields: a multiple of 16 doubles (128 B) so every month row is line aligned."""
    return (int(ncell) + 15) // 16 * 16


def ptr(t):
    return c_void_p(0) if t is None else c_void_p(t.data_ptr())


def as_c(arr, dtype):
    a = np.ascontiguousarray(arr, dtype=dtype)
    ct = {np.float64: c_double, np.int32: c_int, np.int64: c_int64}[dtype]
    return a, a.ctypes.data_as(POINTER(ct))


def dev_vector(arr, dtype=np.float64):
    """Small per-cell vector -> device tensor."""
    torch = torch_cuda()
    if isinstance(arr, torch.Tensor):
        return arr.to(device='cuda', dtype={np.float64: torch.float64, np.int32: torch.int32}[dtype]).contiguous()
    a = np.ascontiguousarray(np.asarray(arr).reshape(-1), dtype=dtype)
    return torch.from_numpy(a).cuda()


class Field:
    """
    A month-major fp64 field resident in HBM: tensor [nmonths, ld], element (m, c) at t[m, c].

    The reference hands [ncell, nmonths] host arrays between its stages; `from_host` / `to_host`
    are the only places where that layout is converted (one transpose kernel each way).
    """

    __slots__ = ('t', 'ncell', 'nmonths')

    def __init__(self, t, ncell):
        self.t = t
        self.ncell = int(ncell)
        self.nmonths = int(t.shape[0])

    @property
    def ld(self):
        return int(self.t.shape[1])

    @classmethod
    def empty(cls, ncell, nmonths, ld=None):
        torch = torch_cuda()
        ld = ld or padded_ld(ncell)
        return cls(torch.empty((nmonths, ld), dtype=torch.float64, device='cuda'), ncell)

    @classmethod
    def from_host(cls, arr, nan_to_num=False, ld=None):
        """[ncell, nmonths] host array (numpy, ideally in pinned memory) or cuda tensor -> Field."""
        torch = torch_cuda()
        if isinstance(arr, Field):
            return arr
        if isinstance(arr, torch.Tensor):
            src = arr.to(device='cuda', dtype=torch.float64, non_blocking=True).contiguous()
        else:
            a = np.asarray(arr)
            if a.dtype != np.float64 or not a.flags['C_CONTIGUOUS']:
                a = np.ascontiguousarray(a, dtype=np.float64)
            src = torch.from_numpy(a).to('cuda', non_blocking=True)
        ncell, nmonths = src.shape
        f = cls.empty(ncell, nmonths, ld)
        check(lib().xan_to_month_major(ptr(src), ptr(f.t), ncell, nmonths, f.ld, int(bool(nan_to_num)), stream_ptr()))
        return f

    def to_device_cell_major(self):
        torch = torch_cuda()
        out = torch.empty((self.ncell, self.nmonths), dtype=torch.float64, device='cuda')
        check(lib().xan_to_cell_major(ptr(self.t), ptr(out), self.ncell, self.nmonths, self.ld, stream_ptr()))
        return out

    def to_host(self):
        """
        Field -> [ncell, nmonths] numpy array.  The host buffer comes from `host_pool` (pinned, recycled when the
        returned array is garbage collected).  Inside `async_host()` the copy runs on a side stream and the array
        must not be read before `host_sync()` (the context manager does that on exit).
        """
        torch = torch_cuda()
        dev = self.to_device_cell_major()
        host = host_pool.acquire((self.ncell, self.nmonths))
        if _async['on']:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            cs = copy_stream('d2h')
            cs.wait_event(ev)
            dev.record_stream(cs)
            with torch.cuda.stream(cs):
                host.copy_(dev, non_blocking=True)
            _async['pending'].append(dev)
        else:
            host.copy_(dev, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return host_pool.as_array(host)


class HostPool:
    """
    Recycling pool of pinned host buffers.  cudaHostAlloc of a 194 MB field costs 50-100 ms, an order of
    magnitude more than the D2H copy it serves (3.4 ms), so buffers are handed out as numpy arrays and taken back
    when those arrays die.  Beyond `limit_bytes` of live pinned memory plain pageable arrays are returned.
    """

    def __init__(self, limit_bytes=24 << 30):
        self.free = {}
        self.live_bytes = 0
        self.limit_bytes = limit_bytes
        self.n_fresh = self.n_reused = self.n_pageable = 0

    def acquire(self, shape):
        torch = torch_cuda()
        n = int(np.prod(shape))
        lst = self.free.get(n)
        if lst:
            self.n_reused += 1
            return lst.pop().view(*shape)
        if self.live_bytes + 8 * n > self.limit_bytes:
            self.n_pageable += 1
            return torch.empty(shape, dtype=torch.float64)
        self.live_bytes += 8 * n
        self.n_fresh += 1
        return torch.empty(shape, dtype=torch.float64, pin_memory=True)

    def reserve(self, shape, count):
        """Makes sure `count` pinned buffers of this size are free in the pool (cudaHostAlloc stalls the device for
        50 - 100 ms per 194 MB field: a pipeline allocates what it will have in flight before it starts)."""
        torch = torch_cuda()
        n = int(np.prod(shape))
        for _ in range(max(0, int(count) - len(self.free.get(n, ())))):
            if self.live_bytes + 8 * n > self.limit_bytes:
                break
            self.live_bytes += 8 * n
            self.n_fresh += 1
            self._release(torch.empty(n, dtype=torch.float64, pin_memory=True))

    def stats(self):
        return dict(fresh=self.n_fresh, reused=self.n_reused, pageable=self.n_pageable, live_bytes=self.live_bytes,
                    free=sum(len(v) for v in self.free.values()))

    def as_array(self, t):
        import weakref
        arr = t.numpy()
        if t.is_pinned():
            weakref.finalize(arr, self._release, t)
        return arr

    def _release(self, t):
        self.free.setdefault(t.numel(), []).append(t.reshape(-1))

    def clear(self):
        self.free.clear()
        self.live_bytes = 0


host_pool = HostPool()
_streams = {}
_async = {'on': False, 'pending': []}


def copy_stream(kind):
    torch = torch_cuda()
    key = (kind, torch.cuda.current_device())
    if key not in _streams:
        _streams[key] = torch.cuda.Stream()
    return _streams[key]


def host_sync():
    """Wait for every asynchronous device->host copy issued under `async_host()`."""
    if _async['pending']:
        copy_stream('d2h').synchronize()
        _async['pending'].clear()


class async_host:
    """
    Context manager: results handed back by the plug-in calls inside the block are copied to the host on a side
    stream while the next stage computes; they are complete when the block exits.
    """

    def __enter__(self):
        self.prev = _async['on']
        _async['on'] = True
        return self

    def __exit__(self, *exc):
        _async['on'] = self.prev
        if not self.prev:
            host_sync()
        return False


def prefetch(host_array, nan_to_num=False):
    """
    Start uploading an input ([ncell, nmonths] host array) on a side stream so that the copy overlaps the
    kernels of an earlier stage; the next `as_field(host_array)` returns the device copy (and makes the compute
    stream wait for it).  The entry is TRANSIENT: it is consumed by that one `as_field` call, because the array
    belongs to the caller, who is free to overwrite it afterwards (see `remember`).
    """
    torch = torch_cuda()
    if host_array is None or isinstance(host_array, Field) or resident(host_array, peek=True) is not None:
        return
    cs = copy_stream('h2d')
    with torch.cuda.stream(cs):
        f = Field.from_host(host_array, nan_to_num=nan_to_num)
        ev = torch.cuda.Event()
        ev.record(cs)
    _register(host_array, f, transient=True, event=ev)


# Device copies of host arrays, so that the next stage of Components.simulation (PET -> runoff -> routing) finds
# its input already in HBM.  Coherence contract (the reference hands plain ndarrays around and its callees mutate
# them, so a stale device copy must never be used silently):
#   * arrays RETURNED by a CUDA stage (`remember`) are handed out READ-ONLY (`flags.writeable = False`): host and
#     device copy cannot diverge.  `res.Q *= 2` raises "output array is read-only"; `q = res.Q * 2` / `res.Q.copy()`
#     are new arrays and are uploaded when they are passed back in.  If an owner re-enables writing
#     (`setflags(write=True)`, possible for arrays that own their memory) the entry is dropped at the next lookup.
#   * arrays OWNED BY THE CALLER (`prefetch`) are trusted for exactly one lookup.
_resident = {}


def _register(host_array, field, transient=False, event=None):
    import weakref
    key = id(host_array)
    _resident[key] = (weakref.ref(host_array, lambda _r, k=key: _resident.pop(k, None)), field, transient, event)


def remember(host_array, field):
    """Register `field` as the device copy of the array a stage returns; the array becomes read-only."""
    try:
        host_array.flags.writeable = False
    except Exception:
        return host_array               # cannot be protected -> not cached
    _register(host_array, field)
    return host_array


def resident(host_array, peek=False):
    """Device copy of `host_array` if it is still known to be identical to it, else None."""
    key = id(host_array)
    hit = _resident.get(key)
    if hit is None or hit[0]() is not host_array:
        return None
    ref, f, transient, ev = hit
    if not transient and getattr(getattr(host_array, 'flags', None), 'writeable', True):
        _resident.pop(key, None)        # the owner made it writeable again: the copies may differ
        return None
    if peek:
        return f
    if transient:
        _resident.pop(key, None)
    if ev is not None:                  # uploaded on the side stream: order the compute stream after it
        cur = torch_cuda().cuda.current_stream()
        cur.wait_event(ev)
        f.t.record_stream(cur)
        if not transient:
            _resident[key] = (ref, f, transient, None)
    return f


def forget_all():
    _resident.clear()


def as_field(x, nan_to_num=False):
    """Field for `x`: an existing Field, the device copy of a previously returned array, or a fresh upload."""
    if x is None:
        return None
    if isinstance(x, Field):
        return x
    f = resident(x)
    if f is not None:
        return f
    return Field.from_host(x, nan_to_num=nan_to_num)
