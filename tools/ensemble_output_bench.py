"""
End-to-end cost of the ensemble runner's output options on the bench world (67,420 cells), alone or under
`torchrun --nproc_per_node N`:

  A  today's default: q + avgchflow monthly grids + basin aggregates
  B  yearly + km3 + basin / country / region sums + mean / std / min / max, member grids copied back (yearly)
  C  as B without member grids (group sums per member, statistics once at the end)
  Q  as C plus the across-member quantiles (0.05, 0.5, 0.95) of every variable
  D  as C plus drought statistics of q with per-member thresholds over the first 30 years (DroughtSpec)

at config-1 length (1971-2000, 360 months) with 20 members per rank, and legs C and D at config 5 (64 members,
2015-2100, 1,032 months).  Forcing values are single precision and cross the link as float32, as in bench.py's end-to-end leg.
Each leg: one warm-up run, then the median of five runs (wall time of run_ensemble, max over ranks; every run listed).
Also measured: the across-member statistics update kernel (xan_ens_stats_update) at config-5 size with CUDA events,
and, on rank 0, that the merged statistics of leg C equal those of all members run by one process.  With leg Q: the
quantile kernel (xan_ens_quantiles) alone over 64 members of yearly (86) and monthly (1,032) fields, CUDA events.
With leg D: the drought scan (xan_drought_scan) alone at config-5 size, accumulation only and with severity /
intensity / duration, CUDA events.
`--legs` picks the legs.

    python tools/ensemble_output_bench.py --out profiles/ensemble_output_n1.json
    python tools/ensemble_output_bench.py --legs C,Q --config5-members 0 --out profiles/ensemble_quantiles_n1.json
    torchrun --nproc_per_node 8 tools/ensemble_output_bench.py --out profiles/ensemble_output_n8.json
"""

import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the bench world and its forcing)

STATS_BYTES_PER_ELEMENT = 72      # read x (8 B), read and write (sum, m2) and (min, max) (2 x 2 x 16 B)


def card():
    import torch
    info = {'name': torch.cuda.get_device_name(), 'count': torch.cuda.device_count()}
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader',
                              '-i', str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = out.stdout.strip()
    except Exception as e:           # the numbers are reported without it, and say so
        info['power_limit_and_max_sm_clock'] = 'unavailable: %s' % e
    return info


def group_ids(world, seed=1):
    """Country and region maps shaped like synthetic.write_example's (0 = no country)."""
    nc, nr = max(2, world.n_basins // 2), max(2, world.n_basins // 3)
    rng = np.random.default_rng(seed + 4242)
    country = (world.basin_ids % (nc + 1)).astype(int)
    country[rng.random(world.ncell) < 0.01] = 0
    return country, (world.basin_ids % nr).astype(int) + 1


def setup(sy, ey):
    """The bench world with the same forcing on every rank (members 2k and 2k + 1 differ), so that the statistics of a
    run over several ranks can be compared with those of one process."""
    import torch
    from xanthos_b200 import synthetic, ensemble as ens
    from xanthos_b200.routing import mrtm
    world = synthetic.make_world(seed=0)
    m = (ey - sy + 1) * 12
    pm = synthetic.pm_inputs(world, sy, ey, nlcs=bench.NLCS, seed=1)
    ab = synthetic.abcd_inputs(world, m, seed=1, with_pet=False)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(np.float32))).pin_memory().numpy()
    mem_a = {k: pin(np.nan_to_num(pm[k])) for k in ens.PM_FORCING}
    mem_a['precip'], mem_a['tmin'] = pin(np.nan_to_num(ab['precip'])), pin(np.nan_to_num(ab['tmin']))
    mem_b = {k: pin(np.roll(v, 11, axis=0)) for k, v in mem_a.items()}
    s = world.settings()
    um = mrtm.upstream_genmatrix(mrtm.upstream(world.coords, mrtm.downstream(world.coords, world.flow_dir, s), s))
    tables = {k: v for k, v in pm.items() if k not in ens.PM_FORCING + ('lct_load', 'tairprev_load')}
    country, region = group_ids(world)
    st = ens.EnsembleStatics(world.ncell, sy, ey, tables, pm['lct_load'], pm['elev'], pm['water_idx'], pm['snow_idx'],
                             pm['lc_years'], bench.NLCS, world.n_basins, world.basin_ids, ab['pars'], world.area,
                             world.flow_dist, world.velocity, um, bench.month_days_mod4(m, sy), bench.DT,
                             min(bench.RUNOFF_SPINUP, m), min(bench.ROUTING_SPINUP, m), country_ids=country,
                             region_ids=region)
    return st, mem_a, mem_b


def time_leg(st, members, kw, world_size, reps):
    import torch
    import torch.distributed as dist
    from xanthos_b200 import ensemble as ens
    sink = []

    def keep(i, r):
        sink.append(len(r))

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ens.run_ensemble(st, members[:4 * world_size], on_result=keep, **kw)
    each, stats = [], None
    for _ in range(reps):
        gc.collect()
        gc.disable()
        try:
            barrier()
            t0 = time.perf_counter()
            er = ens.run_ensemble(st, members, on_result=keep, **kw)
            barrier()
            ms = (time.perf_counter() - t0) * 1e3
        finally:
            gc.enable()
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        each.append(float(t[0]))
        stats = er['stats']
    nloc = max(stats['members_local'], 1)
    med = float(np.median(each))
    return {'ms_median': round(med, 2), 'ms_each_run': [round(v, 2) for v in each], 'members': len(members),
            'members_local_rank0': nloc, 'ms_per_member': round(med / nloc, 2),
            'h2d_bytes_per_member': int(stats['h2d_bytes'] // nloc), 'd2h_bytes_per_member': int(stats['d2h_bytes'] // nloc)}, er


def stats_update_kernel(ncell, ntime, launches=20):
    """xan_ens_stats_update on a [ntime][ld] field at steady state (member count >= 2), CUDA events around `launches`
    back-to-back launches; the working set (x + 32 B of state per element) is far larger than the L2."""
    import torch
    from xanthos_b200 import _cuda as C
    ld = C.padded_ld(ncell)
    x = torch.rand((ntime, ld), dtype=torch.float64, device='cuda')
    sm = torch.empty((ntime, ld, 2), dtype=torch.float64, device='cuda')
    mm = torch.empty_like(sm)
    lib, stream = C.lib(), C.stream_ptr()

    def launch(n):
        C.check(lib.xan_ens_stats_update(C.ptr(x), C.ptr(sm), C.ptr(mm), ncell, ntime, ld, n, stream))
    for n in range(1, 4):
        launch(n)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for n in range(4, 4 + launches):
        launch(n)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / launches
    gbs = STATS_BYTES_PER_ELEMENT * ncell * ntime / (ms * 1e-3) / 1e9
    return {'ncell': ncell, 'ntime': ntime, 'ms_per_launch': round(ms, 4), 'bytes_per_element': STATS_BYTES_PER_ELEMENT,
            'gb_per_s': round(gbs, 1), 'frac_of_6551_gbs_copy_peak': round(gbs / 6551.0, 3), 'target_frac': 0.70}


QUANTILE_LEVELS = (0.05, 0.5, 0.95)


def quantile_kernel(ncell, ntime, n=64, launches=20):
    """xan_ens_quantiles over a member stack [n, ntime, ld] (all of QUANTILE_LEVELS in one launch), CUDA events
    around `launches` back-to-back launches after two warm-up launches; the stack is far larger than the L2.  Bytes
    per second count the stack read once and the cell-major output written once."""
    import torch
    from xanthos_b200 import ensemble as ens, _cuda as C
    ld = C.padded_ld(ncell)
    stack = torch.rand((n, ntime, ld), dtype=torch.float64, device='cuda')
    out = torch.empty((len(QUANTILE_LEVELS), ncell, ntime), dtype=torch.float64, device='cuda')
    for _ in range(2):
        ens.member_quantiles(stack, ncell, QUANTILE_LEVELS, out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        ens.member_quantiles(stack, ncell, QUANTILE_LEVELS, out)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / launches
    read, written = 8 * n * ntime * ncell, 8 * len(QUANTILE_LEVELS) * ntime * ncell
    del stack, out
    torch.cuda.empty_cache()
    return {'members': n, 'ncell': ncell, 'ntime': ntime, 'levels': list(QUANTILE_LEVELS), 'launches': launches,
            'ms_per_launch': round(ms, 3), 'stack_bytes_read': read, 'bytes_written': written,
            'gb_per_s': round((read + written) / (ms * 1e-3) / 1e9, 1)}


DROUGHT_YEARS = 30                # per-member thresholds from the first 30 years of the run, as a 1971-2000 baseline


def drought_spec(sy):
    from xanthos_b200 import ensemble as ens
    return ens.DroughtSpec('q', threshold_years=(sy, sy + DROUGHT_YEARS - 1))


def drought_kernel(ncell, nmonths, launches=20):
    """xan_drought_scan over a [nmonths][ld] field with 12 threshold rows, CUDA events around `launches` back-to-back
    launches after two warm-up launches, accumulation only and accumulation plus severity / intensity / duration.  The
    field and the counts (12 B per cell-month) are far larger than the L2.  Algorithmic bytes per cell-month: the
    field read (8), the count read and written (4 + 4) and with the fields 24 B written; per cell the 12 threshold
    rows read once (96) and the summary written (32)."""
    import torch
    from xanthos_b200 import _cuda as C
    from xanthos_b200.drought.drought_stats import drought_scan_device
    ld = C.padded_ld(ncell)
    g = torch.Generator(device='cuda').manual_seed(5)
    hydro = torch.rand((nmonths, ld), dtype=torch.float64, device='cuda', generator=g)
    th = torch.full((12, ncell), 0.1, dtype=torch.float64, device='cuda')       # about 10 % of the months are dry
    count = torch.zeros((nmonths, ld), dtype=torch.int32, device='cuda')
    summary = torch.empty((4, ld), dtype=torch.float64, device='cuda')
    sid = [torch.empty((nmonths, ld), dtype=torch.float64, device='cuda') for _ in range(3)]
    out = {'ncell': ncell, 'nmonths': nmonths, 'launches': launches, 'dry_fraction': 0.1}
    for name, fields in (('accumulate', None), ('accumulate_and_fields', sid)):
        for _ in range(2):
            drought_scan_device(hydro, ncell, th, fields, count, summary)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            drought_scan_device(hydro, ncell, th, fields, count, summary)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / launches
        nbytes = (16 + (24 if fields else 0)) * ncell * nmonths + (96 + 32) * ncell
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {'ms_per_launch': round(ms, 4), 'algorithmic_bytes': nbytes, 'gb_per_s': round(gbs, 1),
                     'frac_of_6551_gbs_copy_peak': round(gbs / 6551.0, 3)}
    del hydro, count, sid
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--members', type=int, default=20, help='members per rank at config-1 length')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--config5-members', type=int, default=64, help='0 skips the config-5 leg')
    ap.add_argument('--legs', default='A,B,C,Q', help='comma-separated subset of A, B, C, Q, D')
    ap.add_argument('--rounds', type=int, default=1, help='the legs in turn this many times (drift shows between '
                                                          'rounds); the last round is reported per leg')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from xanthos_b200 import ensemble as ens, _cuda as C
    world_size = int(os.environ.get('WORLD_SIZE', '1'))
    rank, local_rank = int(os.environ.get('RANK', '0')), int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    C.lib()
    spec_b = dict(output_in_year=True, output_unit='km3', group_sums=ens.GROUP_SCALES, stats=ens.STATS)
    legs = {'A': dict(), 'B': dict(aggregates=False, spec=ens.OutputSpec(**spec_b)),
            'C': dict(aggregates=False, spec=ens.OutputSpec(member_fields=False, **spec_b)),
            'Q': dict(aggregates=False, spec=ens.OutputSpec(member_fields=False, quantiles=QUANTILE_LEVELS, **spec_b)),
            'D': dict(aggregates=False, spec=ens.OutputSpec(member_fields=False, drought=drought_spec(bench.START_YR),
                                                            **spec_b))}
    legs_order = [k for k in args.legs.split(',') if k in legs]
    legs = {k: legs[k] for k in legs_order}
    out = {'card': card(), 'world_size': world_size, 'transport': 'float32 (single-precision forcing values)',
           'config1': {}, 'config5': {}}

    st, mem_a, mem_b = setup(bench.START_YR, bench.END_YR)
    members = [mem_a if k % 2 == 0 else mem_b for k in range(args.members * world_size)]
    out['config1_rounds'] = []
    for rnd, name in [(r_, n_) for r_ in range(args.rounds) for n_ in legs]:
        out['config1'][name], er = time_leg(st, members, legs[name], world_size, args.reps)
        if name == legs_order[0]:
            out['config1_rounds'].append({})
        out['config1_rounds'][-1][name] = out['config1'][name]['ms_each_run']
        kw = legs[name]
        if name == 'Q' and rank == 0 and rnd == 0:
            # the end-of-run quantile step alone (selection + copy of the result to the host), one process
            r = ens.EnsembleRunner(st, ('q', 'avgchflow'), aggregates=False, spec=kw['spec'])
            for _ in r.run(members):
                pass
            each = []
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r.finalize_quantiles([r.member_stack()])
                each.append(round((time.perf_counter() - t0) * 1e3, 2))
            out['config1']['Q']['finalize_quantiles_ms_each'] = each
            del r
        if name == 'C' and rank == 0 and rnd == 0:
            # the merged statistics against one process running every member (this rank's runner, no exchange)
            r = ens.EnsembleRunner(st, ('q', 'avgchflow'), aggregates=False, spec=kw['spec'])
            for _ in r.run(members):
                pass
            one = r.finalize_stats(r.stats_partial(), len(members))
            dev = {}
            for v in one:
                for s_ in ens.STATS:
                    a, b = er['ensemble_stats'][v][s_], one[v][s_]
                    same_nan = bool(np.array_equal(np.isnan(a), np.isnan(b)))
                    ok = ~np.isnan(b)
                    rel = float(np.max(np.abs(a[ok] - b[ok]) / np.maximum(np.abs(b[ok]), 1e-300))) if ok.any() else 0.0
                    dev['%s.%s' % (v, s_)] = {'bitwise': bool(same_nan and np.array_equal(a[ok], b[ok])),
                                              'max_rel': rel, 'nan_pattern_equal': same_nan}
            out['config1']['C']['merged_vs_single_process'] = dev
        del er
    del st, mem_a, mem_b, members
    gc.collect()
    torch.cuda.empty_cache()
    if rank == 0:
        out['stats_update_kernel_config5'] = stats_update_kernel(bench.NCELL, 1032)
        if 'Q' in legs:
            out['quantile_kernel'] = {'yearly': quantile_kernel(bench.NCELL, 86),
                                      'monthly': quantile_kernel(bench.NCELL, 1032)}
        if 'D' in legs:
            out['drought_kernel_config5'] = drought_kernel(bench.NCELL, 1032)
    c5 = [k for k in ('C', 'D') if k in legs]
    if args.config5_members > 0 and c5:
        st, mem_a, mem_b = setup(2015, 2100)
        members = [mem_a if k % 2 == 0 else mem_b for k in range(args.config5_members)]
        if 'D' in legs:
            legs['D'] = dict(legs['D'], spec=ens.OutputSpec(member_fields=False, drought=drought_spec(2015), **spec_b))
        for name in c5:
            out['config5'][name], _ = time_leg(st, members, legs[name], world_size, args.reps)
    if rank == 0:
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            with open(args.out, 'w') as f:
                f.write(line + '\n')
    if world_size > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
