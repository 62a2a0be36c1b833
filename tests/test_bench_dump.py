"""bench.py --dump-outputs: file per array, dtypes, the seeded row sample and the size limit (host), and on the GPU what each
workload dumps and that two runs with the same arguments write identical files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_dtypes_and_sample(tmp_path):
    rows = torch.arange(3 * bench.DUMP_ROWS, dtype=torch.int64)
    a, b = bench.sample_rows(rows), bench.sample_rows(rows)
    assert torch.equal(a, b) and a.shape == (bench.DUMP_ROWS,) and bool((a[1:] > a[:-1]).all())
    short = torch.ones(5, 3, dtype=torch.float16)
    assert bench.sample_rows(short) is short
    bench.dump_outputs(str(tmp_path), dict(rows=a, feats=short, depth=torch.zeros(4, dtype=torch.float64), loss=1.5))
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert {k: v.dtype for k, v in got.items()} == dict(rows=np.float64, feats=np.float32, depth=np.float64, loss=np.float64)
    assert np.array_equal(got['rows'], a.numpy()) and got['feats'].shape == (5, 3)


def test_dump_outputs_refuses_more_than_the_limit(tmp_path):
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path), dict(big=torch.zeros(bench.DUMP_LIMIT // 4 + 1)))
    assert not os.listdir(tmp_path)


FRAMES = [f'{q}_frame{k}' for k in range(8) for q in ('depth', 'color')]
DUMPED = {'c2': {'pose', 'tracking_loss', 'mapping_loss', 'added_points', 'feature_rows', 'geo_feats', 'col_feats', 'color_decoder'},
          'c4': {'pose', 'tracking_loss'},
          'c1': {'depth', 'uncertainty', 'color'},
          'rerender': {'psnr', 'depth_l1', *FRAMES}}


def _bench_dump(out, config, points):
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--config', config, '--points', str(points), '--steps', '2', '--warmup', '1',
           '--no-cpu-baseline', '--dump-outputs', str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=bench.ROOT)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line['steps'] == 2 and len(line['step_ms']) == 2
    return {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}


@pytest.mark.gpu
@pytest.mark.parametrize('config', sorted(DUMPED))
def test_bench_dump_outputs_repeat_bit_for_bit(tmp_path, config):
    a = _bench_dump(tmp_path / 'a', config, 60000)
    b = _bench_dump(tmp_path / 'b', config, 60000)
    assert set(a) == DUMPED[config]
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64) and np.isfinite(x).all(), name
        assert x.shape == b[name].shape and np.array_equal(x, b[name]), name
    if 'pose' in a:
        assert a['pose'].shape == (7,)
    if 'feature_rows' in a:
        n = a['feature_rows'].shape[0]
        assert 0 < n <= bench.DUMP_ROWS and a['geo_feats'].shape == a['col_feats'].shape == (n, 32)
    if 'depth' in a:
        rays = bench.CONFIGS[config]['rays']
        assert a['depth'].shape == a['uncertainty'].shape == (rays,) and a['color'].shape == (rays, 3)
