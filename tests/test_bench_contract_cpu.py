"""CPU only: the reference arm of bench.py (the oracle port timed on host cores) prints exactly one JSON line with the
contract's keys, and ranks other than 0 stay silent; --dump-outputs keeps to its size limit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, SCD_BENCH_CPU_ROWS='512', **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                          capture_output=True, text=True, env=env, timeout=300)


def _stand_in_checkout(root):
    """A directory laid out like the reference checkout, holding the one function bench.py imports from it."""
    os.makedirs(root / 'local_utils')
    (root / 'local_utils' / 'faster_mix_k_means_pytorch.py').write_text(
        'import torch\n\n\n'
        'def pairwise_distance(data1, data2, batch_size=None):\n'
        '    return torch.cdist(data1, data2) ** 2\n')
    return root


def test_reference_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    r = _run({'SCD_REFERENCE_DIR': str(_stand_in_checkout(tmp_path / 'reference'))})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'ms' and d['higher_is_better'] is False and d['vs_baseline'] is None
    assert d['metric'].startswith('ms per naming round') and d['value'] > 0 and d['ms_per_step'] == d['value']
    assert d['n_gpus'] == 1 and d['steps'] == 1 and d['warmup'] == 0 and d['data'] == 'synthetic' and d['scaling'] == 'strong'
    assert d['config']['workload'].startswith('C2: 127000x768') and 'model' not in d['config']
    cb = d['cpu_baseline']
    # "reference" where the checkout is importable (the E-step then runs the reference's own pairwise_distance), "port" elsewhere
    assert cb['kind'] == 'reference' and cb['kind_detail'] and cb['cores'] >= 1 and cb['value'] == d['value'] and '512 of 127000 rows' in cb['sample']
    assert cb['reference_checkout_present'] is True
    r2 = _run({'SCD_REFERENCE_DIR': str(tmp_path / 'absent')})
    cb2 = json.loads(r2.stdout.strip())['cpu_baseline']
    assert cb2['kind'] == 'port' and cb2['reference_checkout_present'] is False
    assert d['e2e'] == {'value': d['value'], 'unit': 'ms', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2'})
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_dump_outputs_samples_the_same_rows_of_every_per_row_array_under_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    n, k = 5000, 30
    rng = np.random.default_rng(1)
    outputs = dict(labels=rng.integers(0, k, n), inertia=np.array([3.5]), centers=rng.random((k, 16), dtype=np.float32),
                   topk_vals=rng.random((n, 5), dtype=np.float32), topk_idx=rng.integers(0, 1000, (n, 5)),
                   vote_names=rng.integers(-1, 1000, (k, 20)), vote_counts=rng.integers(0, 9, (k, 20)).astype(np.int32))
    bench.dump_outputs(tmp_path / 'all', outputs, n)                  # under the limit: every row, no row_index
    got = {f[:-len('.npy')]: np.load(tmp_path / 'all' / f) for f in os.listdir(tmp_path / 'all')}
    assert sorted(got) == sorted(outputs)
    for name, a in outputs.items():
        assert got[name].dtype == (np.float32 if a.dtype == np.float32 else np.float64) and np.array_equal(got[name], a)
    monkeypatch.setattr(bench, 'DUMP_BYTES', 100_000)
    for d in ('s1', 's2'):
        bench.dump_outputs(tmp_path / d, outputs, n)
    s1, s2 = ({f[:-len('.npy')]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)} for d in ('s1', 's2'))
    assert sum(a.nbytes for a in s1.values()) <= 100_000
    rows = s1['row_index'].astype(np.int64)
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0) and np.array_equal(s1['row_index'], s2['row_index'])
    for name in ('labels', 'topk_vals', 'topk_idx'):
        assert np.array_equal(s1[name], outputs[name][rows])
    for name in ('centers', 'inertia', 'vote_names', 'vote_counts'):
        assert np.array_equal(s1[name], outputs[name])
    monkeypatch.setattr(bench, 'DUMP_BYTES', 1000)                    # the per-cluster arrays alone are over the limit
    with pytest.raises(ValueError, match='limit'):
        bench.dump_outputs(tmp_path / 'none', outputs, n)
