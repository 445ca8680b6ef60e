"""bench.py --dump-outputs: what the last timed step computed, written as .npy files that two builds can be compared on."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    bench.dump_outputs(str(tmp_path / 'out'), dict(loss=np.ones(1, np.float32), ids=np.arange(3, dtype=np.int32)))
    assert np.load(tmp_path / 'out' / 'loss.npy').dtype == np.float32
    ids = np.load(tmp_path / 'out' / 'ids.npy')
    assert ids.dtype == np.float64 and np.array_equal(ids, [0, 1, 2])
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / 'big'), dict(a=np.zeros(bench.DUMP_LIMIT_BYTES // 8 + 1)))
    assert not (tmp_path / 'big').exists()


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '0'], capture_output=True, text=True)
    assert r.returncode == 2 and '--steps' in r.stderr


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--workload', 'C1', '--steps', str(steps), '--warmup', '1',
           '--no-extras', '--no-cpu-baseline', '--no-e2e', '--dump-outputs', out]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dump_is_reproducible(lib, tmp_path):
    """two runs with the same arguments write the same arrays, bit for bit (no floating-point atomics on the path)"""
    a, b = str(tmp_path / 'a'), str(tmp_path / 'b')
    line = _bench(a, 2)
    assert line['steps'] == 2
    _bench(b, 2)
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    for n in ('loss.npy', 'probs.npy', 'weight_conv_w.npy', 'user_emb_rows.npy', 'user_emb_row_ids.npy'):
        assert n in names, n
    total = 0
    for n in names:
        x, y = np.load(os.path.join(a, n)), np.load(os.path.join(b, n))
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, y), n
        total += x.nbytes
    assert total <= bench.DUMP_LIMIT_BYTES
    assert abs(float(np.load(os.path.join(a, 'loss.npy'))[0]) - line['loss']) < 1e-6
    assert np.load(os.path.join(a, 'probs.npy')).shape == (64, 5)
