"""Host-side tests of the ensemble output options: the numpy restatement of the across-member statistics kernels
against numpy itself, its merge, OutputSpec, and the rank-order fold of partial statistics under gloo."""

import os
import subprocess
import sys

import numpy as np
import pytest

from util import bitwise_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stack(n, seed=0, shape=(37, 29)):
    rng = np.random.default_rng(seed)
    x = rng.normal(50.0, 20.0, (n,) + shape) * rng.uniform(0.1, 10.0, shape)
    x[:, 3, :] = x[0, 3, :]                              # identical members: std exactly 0
    x[rng.integers(0, n), rng.random(shape) < 0.05] = np.nan     # NaN in one member only
    x[:, 5, 7] = np.nan                                  # NaN in every member
    return x


@pytest.mark.filterwarnings("ignore:Degrees of freedom")     # numpy.std of one member with ddof = 1: NaN
@pytest.mark.parametrize("n", [1, 2, 5, 9])
def test_oracle_stats_equal_numpy(n):
    """mean / min / max of the member-order fold are bitwise numpy over the stacked members (NaN propagates like
    numpy.min / numpy.max); std is numpy.std within 1e-12 for ddof 0 and 1."""
    from oracle import ensemble_stats as es
    x = _stack(n, seed=n)
    with np.errstate(invalid='ignore', divide='ignore'):
        for ddof in (0, 1):
            got = es.run(list(x), ddof=ddof)
            assert bitwise_equal(got['mean'], np.mean(x, axis=0))
            assert bitwise_equal(got['min'], np.min(x, axis=0)) and bitwise_equal(got['max'], np.max(x, axis=0))
            want = np.std(x, axis=0, ddof=ddof)
            assert np.array_equal(np.isnan(got['std']), np.isnan(want))
            ok = np.isfinite(want)
            np.testing.assert_allclose(got['std'][ok], want[ok], rtol=1e-12, atol=1e-12 * np.nanmax(np.abs(x)))


@pytest.mark.parametrize("split", [[3, 2], [1, 4], [2, 2, 3]])
def test_oracle_split_and_merge_equals_the_unsplit_fold(split):
    """Partials of contiguous member blocks merged in order (Chan et al.) give the statistics of one fold over all
    members: min / max bitwise, mean and std to the last bits."""
    from oracle import ensemble_stats as es
    x = _stack(sum(split), seed=7)
    whole = es.run(list(x), ddof=1)
    acc, n, k = None, 0, 0
    for m in split:
        part = None
        for j in range(m):
            part = es.update(part, x[k + j], j + 1)
        acc = part if acc is None else es.merge(acc, n, part, m)
        n, k = n + m, k + m
    got = es.finalize(acc, n, ddof=1)
    assert bitwise_equal(got['min'], whole['min']) and bitwise_equal(got['max'], whole['max'])
    for st in ('mean', 'std'):
        assert np.array_equal(np.isnan(got[st]), np.isnan(whole[st]))
        ok = ~np.isnan(whole[st])
        np.testing.assert_allclose(got[st][ok], whole[st][ok], rtol=1e-12, atol=1e-12 * np.nanmax(np.abs(x)))


def test_output_spec_validation_and_from_settings(tmp_path):
    from xanthos_b200 import synthetic, _cuda as C
    from xanthos_b200.ensemble import OutputSpec
    from xanthos_b200.data_reader.ini_reader import ConfigReader
    s = OutputSpec()
    assert (s.output_in_year, s.output_unit, s.group_sums, s.member_fields, s.stats, s.ddof) == (False, 'mm', (), True,
                                                                                                  (), 0)
    for bad in (dict(output_unit='m3'), dict(group_sums=('basin', 'continent')), dict(stats=('median',)),
                dict(stats=('mean', 'mean')), dict(ddof=-1), dict(ddof=0.5)):
        with pytest.raises(C.ValidationException):
            OutputSpec(**bad)
    w = synthetic.make_world(12, 24, 150, 4, seed=3)
    ini, _ = synthetic.write_example(str(tmp_path / 'a'), w, 2001, 2002)
    s = OutputSpec.from_settings(ConfigReader(ini))
    assert (s.output_in_year, s.output_unit, s.group_sums, s.member_fields, s.stats) == (False, 'mm', ('basin',), True, ())
    ini, _ = synthetic.write_example(str(tmp_path / 'b'), w, 2001, 2002, project_overrides={
        'OutputInYear': 1, 'OutputUnit': 1, 'AggregateRunoffBasin': 0, 'AggregateRunoffCountry': 1,
        'AggregateRunoffGCAMRegion': 1})
    s = OutputSpec.from_settings(ConfigReader(ini), member_fields=False, stats=('mean', 'std'), ddof=1)
    assert (s.output_in_year, s.output_unit, s.group_sums) == (True, 'km3', ('country', 'region'))
    assert (s.member_fields, s.stats, s.ddof) == (False, ('mean', 'std'), 1)


FOLD_WORKER = r'''
import sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from xanthos_b200 import sharding
from oracle import ensemble_stats as es
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%s' % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
r = dist.get_rank()
rng = np.random.default_rng(11)
x = rng.normal(3.0, 2.0, (5, 6, 8))
x[4, 2, 3] = np.nan
parts = sharding.partition_members(5, 2)
counts = [len(p) for p in parts]
part = None
for j, k in enumerate(parts[r]):
    part = es.update(part, x[k], j + 1)

def merge(a, na, b, nb):     # the oracle's merge on the tensors the fold moves around
    return [torch.from_numpy(v) for v in es.merge([t.numpy() for t in a], na, [t.numpy() for t in b], nb)]

got = sharding.fold_to_rank0([torch.from_numpy(np.ascontiguousarray(v)) for v in part], counts, merge)
if r == 0:
    p0 = None
    for j in range(3):
        p0 = es.update(p0, x[j], j + 1)
    p1 = es.update(es.update(None, x[3], 1), x[4], 2)
    want = es.merge(p0, 3, p1, 2)
    assert all(np.array_equal(g.numpy(), w, equal_nan=True) for g, w in zip(got, want))
    assert np.isnan(got[0].numpy()[2, 3]) and np.isnan(got[2].numpy()[2, 3])
else:
    assert got is None
dist.destroy_process_group()
print("rank", r, "ok")
'''


def test_two_rank_fold_of_partial_stats_with_gloo(tmp_path):
    """sharding.fold_to_rank0 under a 2-rank gloo group with the oracle's merge: rank 0 holds exactly the serial
    rank-order fold (members {0, 1, 2} on rank 0, {3, 4} on rank 1), the other rank nothing."""
    script = tmp_path / 'worker.py'
    script.write_text(FOLD_WORKER)
    port = str(31500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all('ok' in o for o in outs), outs
