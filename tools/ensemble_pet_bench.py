"""
End-to-end cost of the ensemble runner with each PET model, with and without routing, on the bench world (67,420
cells), alone or under `torchrun --nproc_per_node N`:

  PM    PM -> ABCD -> MRTM, 1971-2000, q + avgchflow grids and basin aggregates (ensemble_output_bench.py leg A, run in
        the same call to show the PM path unchanged)
  HS    HS -> ABCD, no routing, 2006-2100 (BASELINE config 2), tmin the same array as hs_tmin, q grids + basin
        aggregates
  HS-C  as HS with OutputSpec(output_in_year=True, output_unit='km3', member_fields=False, stats=STATS), no aggregates
        (ensemble_output_bench.py leg C)
  HS-R  HS -> ABCD -> MRTM, 1971-2000, q + avgchflow grids and basin aggregates (pairs routed by one launch)
  TH    Thornthwaite -> ABCD, no routing, 2006-2100, q grids + basin aggregates

Forcing values are single precision and cross the link as float32; 20 members per rank, two different members
alternating.  Each leg: one warm-up run, then the median of five runs (ensemble_output_bench.time_leg: wall time of
run_ensemble, max over ranks, every run listed).  The host -> device rate of one pinned float32 field is measured in
the same call (CUDA events), and every leg reports its upload time per member at that rate: a run without routing is
bounded by it.  `--timeline HS,TH` adds one run per named leg with XANTHOS_ENSEMBLE_TIMELINE=1 after the timed runs and
prints its per-member intervals for tools/ensemble_timeline_report.py.

    python tools/ensemble_pet_bench.py --out profiles/ensemble_pet_n1.json
    torchrun --nproc_per_node 8 tools/ensemble_pet_bench.py --out profiles/ensemble_pet_n8.json
"""

import argparse
import gc
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import bench  # noqa: E402  (the bench world's constants)
from ensemble_output_bench import card, setup, time_leg  # noqa: E402

FUTURE = (2006, 2100)                   # BASELINE config 2: 1,140 months
FUTURE_RUNOFF_SPINUP = 360


def pinned32(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).pin_memory().numpy()


def second_member(mem):
    """A different member (cells rolled by 11) with the same arrays shared as in `mem`."""
    rolled = {}
    return {k: rolled.setdefault(id(a), pinned32(np.roll(a, 11, axis=0))) for k, a in mem.items()}


def hs_leg(world, sy, ey, routing, um=None):
    """Statics and two members of HS forcing as DataLoader hands it out (NaN kept in hs_* and precip), tmin the very
    array of hs_tmin."""
    from xanthos_b200 import synthetic
    hs = synthetic.hs_inputs(world, sy, ey, seed=2)
    ab = synthetic.abcd_inputs(world, (ey - sy + 1) * 12, seed=1, with_pet=False)
    mem = {k: pinned32(hs[k]) for k in ('hs_tas', 'hs_tmax', 'hs_tmin')}
    mem['precip'], mem['tmin'] = pinned32(ab['precip']), mem['hs_tmin']
    return statics(world, 'hs', sy, ey, ab['pars'], routing, um), mem, second_member(mem)


def th_leg(world, sy, ey):
    """Statics (no routing) and two members of Thornthwaite forcing as DataLoader hands it out (tair and tmin with NaN
    as 0, NaN kept in precip)."""
    from xanthos_b200 import synthetic
    tw = synthetic.thornthwaite_inputs(world, sy, ey, seed=5)
    ab = synthetic.abcd_inputs(world, (ey - sy + 1) * 12, seed=1, with_pet=False)
    mem = {'tair': pinned32(np.nan_to_num(tw['tair'])), 'precip': pinned32(ab['precip']),
           'tmin': pinned32(np.nan_to_num(ab['tmin']))}
    return statics(world, 'thornthwaite', sy, ey, ab['pars'], False), mem, second_member(mem)


def statics(world, pet, sy, ey, pars, routing, um=None):
    from xanthos_b200 import ensemble as ens
    m = (ey - sy + 1) * 12
    kw = dict(pet=pet, latitude=world.coords[:, 2], routing=routing)
    if routing:
        return ens.EnsembleStatics(world.ncell, sy, ey, None, None, None, None, None, None, None, world.n_basins,
                                   world.basin_ids, pars, world.area, world.flow_dist, world.velocity, um,
                                   bench.month_days_mod4(m, sy), bench.DT, min(bench.RUNOFF_SPINUP, m),
                                   min(bench.ROUTING_SPINUP, m), **kw)
    return ens.EnsembleStatics(world.ncell, sy, ey, None, None, None, None, None, None, None, world.n_basins,
                               world.basin_ids, pars, world.area, None, None, None, None,
                               runoff_spinup=min(FUTURE_RUNOFF_SPINUP, m), **kw)


def h2d_rate(ncell, nmonths, copies=10):
    """GB/s of one pinned float32 [ncell, nmonths] field copied to the device, CUDA events around `copies` copies
    after two warm-up copies."""
    import torch
    src = torch.from_numpy(np.ones((ncell, nmonths), dtype=np.float32)).pin_memory()
    dst = torch.empty(src.shape, dtype=torch.float32, device='cuda')
    for _ in range(2):
        dst.copy_(src, non_blocking=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(copies):
        dst.copy_(src, non_blocking=True)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / copies
    return {'bytes': src.numel() * 4, 'copies': copies, 'ms_per_copy': round(ms, 3),
            'gb_per_s': round(src.numel() * 4 / (ms * 1e-3) / 1e9, 2)}


def timeline(st, members, kw):
    """One run with XANTHOS_ENSEMBLE_TIMELINE=1: per member (h2d start, end), (compute start, end), outputs on the
    host, ms since the first upload."""
    from xanthos_b200 import ensemble as ens
    os.environ['XANTHOS_ENSEMBLE_TIMELINE'] = '1'
    try:
        tl = ens.run_ensemble(st, members, on_result=lambda i, r: None, **kw)['stats'].get('timeline')
    finally:
        del os.environ['XANTHOS_ENSEMBLE_TIMELINE']
    print('ensemble timeline (ms since the first upload): %s' % json.dumps(tl), flush=True)
    return tl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--members', type=int, default=20, help='members per rank')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--legs', default='PM,HS,HS-C,HS-R,TH')
    ap.add_argument('--timeline', default='', help='legs that get one extra run with XANTHOS_ENSEMBLE_TIMELINE=1')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from xanthos_b200 import synthetic, ensemble as ens, _cuda as C
    from xanthos_b200.routing import mrtm
    world_size = int(os.environ.get('WORLD_SIZE', '1'))
    rank, local_rank = int(os.environ.get('RANK', '0')), int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    C.lib()
    wanted = args.legs.split(',')
    world = synthetic.make_world(seed=0)
    n_future = (FUTURE[1] - FUTURE[0] + 1) * 12
    out = {'card': card(), 'world_size': world_size, 'transport': 'float32 (single-precision forcing values)',
           'members_per_rank': args.members, 'h2d_one_field': h2d_rate(world.ncell, n_future), 'legs': {}}
    rate = out['h2d_one_field']['gb_per_s']
    past = (bench.START_YR, bench.END_YR)
    um = None
    if 'HS-R' in wanted:
        s = world.settings()
        um = mrtm.upstream_genmatrix(mrtm.upstream(world.coords, mrtm.downstream(world.coords, world.flow_dir, s), s))
    hs_c = ens.OutputSpec(output_in_year=True, output_unit='km3', member_fields=False, stats=ens.STATS)
    # leg -> (what it runs, statics and members (made when the leg runs), runner arguments)
    legs = {
        'PM': ('PM -> ABCD -> MRTM, %d-%d, q + avgchflow grids + basin aggregates' % past,
               lambda: setup(*past), dict()),
        'HS': ('HS -> ABCD, no routing, %d-%d, tmin is hs_tmin, q grids + basin aggregates' % FUTURE,
               lambda: hs_leg(world, *FUTURE, False), dict(output_vars=('q',))),
        'HS-C': ('as HS, OutputSpec(output_in_year=True, output_unit=km3, member_fields=False, stats=STATS), '
                 'no aggregates', None, dict(output_vars=('q',), aggregates=False, spec=hs_c)),
        'HS-R': ('HS -> ABCD -> MRTM, %d-%d, q + avgchflow grids + basin aggregates' % past,
                 lambda: hs_leg(world, *past, True, um), dict()),
        'TH': ('Thornthwaite -> ABCD, no routing, %d-%d, q grids + basin aggregates' % FUTURE,
               lambda: th_leg(world, *FUTURE), dict(output_vars=('q',))),
    }
    made = members = None
    for name in [k for k in legs if k in wanted]:
        what, make, kw = legs[name]
        if make is not None or made is None:      # HS-C runs on the statics and members of HS
            made = members = None
            gc.collect()
            made = (make or legs['HS'][1])()
        st, mem_a, mem_b = made
        members = [mem_a if k % 2 == 0 else mem_b for k in range(args.members * world_size)]
        res, _ = time_leg(st, members, kw, world_size, args.reps)
        uniq = len({id(a) for a in mem_a.values()})
        res['fields_uploaded_per_member'] = uniq
        res['h2d_bytes_per_member_expected'] = uniq * st.ncell * st.nmonths * 4
        res['upload_ms_per_member'] = round(res['h2d_bytes_per_member'] / (rate * 1e9) * 1e3, 2)
        res['ms_per_member_over_upload'] = round(res['ms_per_member'] / res['upload_ms_per_member'], 3)
        out['legs'][name] = dict(runs=what, nmonths=st.nmonths, **res)
        if name in args.timeline.split(','):
            tl = timeline(st, members, kw)
            if rank == 0:
                out['legs'][name]['timeline'] = tl
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
