"""
Parameter ensembles (one forcing, many ABCD parameter tables) on the bench world (67,420 cells), one GPU:

  kernel  one xan_abcd_run_sets call of S tables against S calls of xan_abcd_run over the same month-major forcing,
          S = 1, 2, 4, 8, 1971-2000 with snow (tmin given), 360 months of spin-up: CUDA events around each side, the two
          alternating in one process, `--kernel-reps` times each after one warm-up of each; the median per set.  The
          outputs of the two sides are compared bit for bit in the same run.  This is the measurement behind the sets
          per thread (ABCD_SETS_PER_THREAD, csrc/abcd.cu) and ensemble.PARAMETER_SETS_PER_LAUNCH.
  PM      PM -> ABCD -> MRTM, 1971-2000, 20 sets, q + avgchflow grids and basin aggregates: run_parameter_ensemble
          against run_ensemble over the same forcing given 20 times
  HS      HS -> ABCD, no routing, 2006-2100, 64 sets, OutputSpec(output_in_year=True, output_unit='km3',
          member_fields=False, stats=STATS), q, no aggregates: the same comparison

The end-to-end legs: one warm-up run of each side, then five runs of each, alternating; wall time of the call (ending
in a device synchronise), every run listed, the median per set.  Forcing values are single precision and cross the
link as float32, as in tools/ensemble_pet_bench.py.  The parameter tables are the world's table scaled per entry by
factors in [0.9, 1] (seeded).  The card's name and power limit are read in the same call.

    python tools/parameter_ensemble_bench.py --out profiles/parameter_ensemble_n1.json
"""

import argparse
import gc
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import bench  # noqa: E402  (the bench world's constants)
from ensemble_output_bench import card, setup  # noqa: E402
from ensemble_pet_bench import FUTURE, hs_leg  # noqa: E402


def tables(pars, n, seed=3):
    """n parameter tables [n, rows, 5]: the first is `pars`, the others scale every entry by a factor in [0.9, 1]."""
    rng = np.random.default_rng(seed)
    out = np.repeat(np.asarray(pars, dtype=np.float64)[None], n, axis=0)
    out[1:] *= rng.uniform(0.9, 1.0, out[1:].shape)
    return out


def kernel_leg(world, sets=(1, 2, 4, 8), reps=20):
    """Per-set ms of one xan_abcd_run_sets call of S tables and of S xan_abcd_run calls, and their bitwise equality."""
    import torch
    from xanthos_b200 import synthetic, _cuda as C
    from xanthos_b200.runoff import abcd
    m = bench.NMONTHS
    ab = synthetic.abcd_inputs(world, m, seed=1, with_pet=True)
    rows = abcd._basin_rows(world.n_basins, world.basin_ids, ab['pars'].shape[0])
    plan = abcd.basin_plan(rows, world.n_basins)
    e, p, t = (C.Field.from_host(ab[k], nan_to_num=(k == 'tmin')) for k in ('pet', 'precip', 'tmin'))
    pars = torch.from_numpy(tables(ab['pars'], max(sets))).cuda()
    n_rows, ld, L = int(pars.shape[1]), e.ld, C.lib()
    outs = {side: [[torch.empty((m, ld), dtype=torch.float64, device='cuda') for _ in range(3)]
                   for _ in range(max(sets))] for side in ('sets', 'single')}

    def run_sets(S):
        arr = [(C.c_void_p * S)(*[outs['sets'][k][i].data_ptr() for k in range(S)]) for i in range(3)]
        C.check(L.xan_abcd_run_sets(plan._plan, S, n_rows, C.ptr(e.t), C.ptr(p.t), C.ptr(t.t), C.ptr(pars), m,
                                    bench.RUNOFF_SPINUP, ld, arr[0], arr[1], arr[2], C.stream_ptr()))

    def run_single(S):
        for k in range(S):
            o = outs['single'][k]
            C.check(L.xan_abcd_run(plan._plan, C.ptr(e.t), C.ptr(p.t), C.ptr(t.t), C.ptr(pars[k]), m,
                                   bench.RUNOFF_SPINUP, ld, C.ptr(o[0]), C.ptr(o[1]), C.ptr(o[2]), C.stream_ptr()))

    def timed(fn, S):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(S)
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    res = {}
    for S in sets:
        run_sets(S)
        run_single(S)
        ms = {'sets': [], 'single': []}
        for _ in range(reps):
            ms['sets'].append(timed(run_sets, S))
            ms['single'].append(timed(run_single, S))
        torch.cuda.synchronize()
        same = all(torch.equal(outs['sets'][k][i][:, :world.ncell].view(torch.int64),
                               outs['single'][k][i][:, :world.ncell].view(torch.int64))
                   for k in range(S) for i in range(3))
        med = {k: float(np.median(v)) / S for k, v in ms.items()}
        res[str(S)] = {'ms_per_set_run_sets': round(med['sets'], 3), 'ms_per_set_run': round(med['single'], 3),
                       'run_sets_over_run': round(med['sets'] / med['single'], 4), 'bitwise_equal': bool(same),
                       'ms_each_call_run_sets': [round(v, 3) for v in ms['sets']],
                       'ms_each_s_calls_run': [round(v, 3) for v in ms['single']]}
        print('kernel S=%d: %s' % (S, json.dumps({k: v for k, v in res[str(S)].items() if 'each' not in k})),
              flush=True)
    return {'nmonths': m, 'spinup': bench.RUNOFF_SPINUP, 'ncell': world.ncell, 'reps': reps, 'snow': True,
            'sets': res}


def e2e_leg(st, forcing, sets, kw, reps=5):
    """Median wall ms per set of run_parameter_ensemble(st, forcing, sets) and of run_ensemble(st, [forcing] * P)."""
    import torch
    from xanthos_b200 import ensemble as ens
    n = len(sets)
    side = {'run_parameter_ensemble': lambda: ens.run_parameter_ensemble(st, forcing, sets, on_result=sink, **kw),
            'run_ensemble': lambda: ens.run_ensemble(st, [forcing] * n, on_result=sink, **kw)}

    def sink(i, r):
        pass
    for fn in side.values():
        fn()
    each, stats = {k: [] for k in side}, {}
    for _ in range(reps):
        for k, fn in side.items():
            gc.collect()
            gc.disable()
            try:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = fn()
                torch.cuda.synchronize()
                each[k].append((time.perf_counter() - t0) * 1e3)
            finally:
                gc.enable()
            stats[k] = r['stats']
    out = {'sets': n}
    for k in side:
        med = float(np.median(each[k]))
        out[k] = {'ms_median': round(med, 2), 'ms_each_run': [round(v, 2) for v in each[k]],
                  'ms_per_set': round(med / n, 2), 'h2d_bytes': int(stats[k]['h2d_bytes']),
                  'd2h_bytes': int(stats[k]['d2h_bytes'])}
    out['speedup_per_set'] = round(out['run_ensemble']['ms_per_set'] / out['run_parameter_ensemble']['ms_per_set'], 3)
    print('%s' % json.dumps({k: (v if not isinstance(v, dict) else {a: b for a, b in v.items() if a != 'ms_each_run'})
                             for k, v in out.items()}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--legs', default='kernel,PM,HS')
    ap.add_argument('--kernel-reps', type=int, default=20)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from xanthos_b200 import synthetic, ensemble as ens, _cuda as C
    C.lib()
    if not torch.cuda.is_available():
        raise SystemExit("parameter_ensemble_bench needs a CUDA device")
    wanted = args.legs.split(',')
    world = synthetic.make_world(seed=0)
    out = {'card': card(), 'legs': {}}
    if 'kernel' in wanted:
        out['legs']['kernel'] = kernel_leg(world, reps=args.kernel_reps)
    if 'PM' in wanted:
        st, mem, _ = setup(bench.START_YR, bench.END_YR)
        leg = e2e_leg(st, mem, tables(np.asarray(st.d_pars.cpu()), 20), dict(), args.reps)
        out['legs']['PM'] = dict(runs='PM -> ABCD -> MRTM, %d-%d, q + avgchflow grids + basin aggregates'
                                 % (bench.START_YR, bench.END_YR), nmonths=st.nmonths, **leg)
        del st, mem
        gc.collect()
    if 'HS' in wanted:
        st, mem, _ = hs_leg(world, *FUTURE, False)
        spec = ens.OutputSpec(output_in_year=True, output_unit='km3', member_fields=False, stats=ens.STATS)
        leg = e2e_leg(st, mem, tables(np.asarray(st.d_pars.cpu()), 64), dict(output_vars=('q',), aggregates=False,
                                                                            spec=spec), args.reps)
        out['legs']['HS'] = dict(runs='HS -> ABCD, no routing, %d-%d, OutputSpec(output_in_year=True, output_unit=km3, '
                                 'member_fields=False, stats=STATS), q, no aggregates' % FUTURE, nmonths=st.nmonths,
                                 **leg)
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
