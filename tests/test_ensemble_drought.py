"""Host-side tests of the ensemble runner's drought statistics: DroughtSpec / OutputSpec(drought=...) validation and
from_settings, and the rank-order fold of the drought counts under gloo."""

import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_drought_spec_refusals():
    from xanthos_b200 import _cuda as C
    from xanthos_b200.ensemble import DroughtSpec, OutputSpec
    with pytest.raises(C.ValidationException, match='drought variable'):
        DroughtSpec('runoff', threshold_years=(2001, 2002))
    with pytest.raises(C.ValidationException, match='one of the two'):
        DroughtSpec('q')
    with pytest.raises(C.ValidationException, match='one of the two'):
        DroughtSpec('q', thresholds=np.ones((12, 5)), threshold_years=(2001, 2002))
    with pytest.raises(C.ValidationException):
        DroughtSpec('q', thresholds=np.ones(5))
    with pytest.raises(C.ValidationException):
        DroughtSpec('q', threshold_years=(2001, 2002), nper=0)
    with pytest.raises(C.ValidationException):
        OutputSpec(drought={'var': 'q'})
    # a threshold array whose cell count is wrong
    with pytest.raises(C.ValidationException, match='4 cells, the run 5'):
        DroughtSpec('q', thresholds=np.ones((12, 4))).validate(5, 2001, 2003)
    DroughtSpec('q', thresholds=np.ones((3, 5))).validate(5, 2001, 2003)
    # threshold years outside the run
    for years in ((2000, 2002), (2002, 2004)):
        with pytest.raises(C.ValidationException, match='outside the run'):
            DroughtSpec('soilmoisture', threshold_years=years).validate(5, 2001, 2003)
    # the reference's slice [(sy - start) * 12 : (ey + 1 - sy) * 12] is empty, or not a multiple of nper
    with pytest.raises(C.ValidationException, match='give 0 months'):
        DroughtSpec('q', threshold_years=(2003, 2003)).validate(5, 2001, 2003)       # [24:12]
    with pytest.raises(C.ValidationException, match='give 0 months'):
        DroughtSpec('q', threshold_years=(2002, 2001)).validate(5, 2001, 2003)
    with pytest.raises(C.ValidationException, match='not a positive multiple of 5'):
        DroughtSpec('q', threshold_years=(2001, 2003), nper=5).validate(5, 2001, 2003)
    s = DroughtSpec('Q', threshold_years=(2002, 2003))                              # [12:24]
    assert s.var == 'q' and s.reference_months(2001, 2003) == (12, 24)
    assert DroughtSpec('q', threshold_years=(2001, 2003), nper=4).reference_months(2001, 2003) == (0, 36)


def _example(tmp_path, name, drought):
    from xanthos_b200 import synthetic
    w = synthetic.make_world(12, 24, 150, 4, seed=3)
    ini, _ = synthetic.write_example(str(tmp_path / name), w, 2001, 2003,
                                     postproc={'drought': drought} if drought else None, project_overrides={'OutputInYear': 1, 'OutputUnit': 1})
    return w, ini


def test_from_settings_drought_section(tmp_path):
    from xanthos_b200 import _cuda as C
    from xanthos_b200.ensemble import OutputSpec
    from xanthos_b200.data_reader.ini_reader import ConfigReader
    w, ini = _example(tmp_path, 'years', {'drought_var': 'soilmoisture', 'threshold_nper': 6,
                                          'threshold_start_year': 2001, 'threshold_end_year': 2002})
    cfg = ConfigReader(ini)
    s = OutputSpec.from_settings(cfg, member_fields=False, drought=True)
    d = s.drought
    assert (d.var, d.thresholds, d.threshold_years, d.nper, d.fields) == ('soilmoisture', None, (2001, 2002), 6, False)
    assert (s.output_in_year, s.output_unit, s.member_fields) == (True, 'km3', False)
    assert repr(s).endswith(", drought=DroughtSpec(var='soilmoisture', threshold_years=(2001, 2002), nper=6, "
                            "fields=False))")
    # without drought=True the spec is exactly what it was before the option existed
    plain = OutputSpec.from_settings(cfg, member_fields=False)
    assert plain.drought is None
    assert repr(plain) == ("OutputSpec(output_in_year=True, output_unit='km3', group_sums=('basin',), "
                           "member_fields=False, stats=(), ddof=0, quantiles=())")

    th = np.random.default_rng(2).random((12, w.ncell))
    path = str(tmp_path / 'thresholds.npy')
    np.save(path, th)
    _, ini = _example(tmp_path, 'file', {'drought_var': 'q', 'drought_thresholds': path})
    d = OutputSpec.from_settings(ConfigReader(ini), drought=True).drought
    assert d.var == 'q' and d.threshold_years is None and np.array_equal(d.thresholds, th)
    d.validate(w.ncell, 2001, 2003)
    assert 'thresholds=<12 x {}>'.format(w.ncell) in repr(d)

    _, ini = _example(tmp_path, 'none', None)
    cfg = ConfigReader(ini)
    with pytest.raises(C.ValidationException, match=r'\[Drought\]'):
        OutputSpec.from_settings(cfg, drought=True)
    assert OutputSpec.from_settings(cfg).drought is None


FOLD_WORKER = r'''
import sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from xanthos_b200 import sharding
from xanthos_b200.ensemble import merge_drought_counts
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%s' % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
r = dist.get_rank()
counts = [int(c) for c in sys.argv[4].split(',')]
nmonths, ld = 37, 16
rng = np.random.default_rng(7)
dry = rng.random((sum(counts), nmonths, ld)) < 0.4              # member k is in drought at (t, c)
o = sum(counts[:r])
mine = dry[o:o + counts[r]].sum(axis=0).astype(np.int32)     # what this rank's runner counted
partial = [torch.from_numpy(mine)] if counts[r] or r == 0 else None
got = sharding.fold_to_rank0(partial, counts, merge_drought_counts)
if r == 0:
    want = dry.sum(axis=0).astype(np.int32)
    assert got[0].dtype == torch.int32 and np.array_equal(got[0].numpy(), want)
else:
    assert got is None
dist.destroy_process_group()
print("rank", r, "ok")
'''


@pytest.mark.parametrize("counts", ["3,2", "4,0", "0,4"])
def test_two_rank_fold_of_drought_counts_with_gloo(tmp_path, counts):
    """sharding.fold_to_rank0 with merge_drought_counts under a 2-rank gloo group: rank 0 holds the exact integer sum
    of the members in drought (a rank without members contributes zeros or nothing)."""
    script = tmp_path / 'worker.py'
    script.write_text(FOLD_WORKER)
    port = str(35700 + (os.getpid() * 5 + len(counts) + int(counts[0])) % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r), counts], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all('ok' in o for o in outs), outs
