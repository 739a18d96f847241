"""bench.py --dump-outputs: two runs with the same arguments write the same arrays (the fp32 centres and inertia within
the 1e-5 their run-to-run variation stays under), and what they hold is the round from the initial centroids that the
`parity` hashes of the JSON line describe."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from scd_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--config', 'C1', '--steps', '3', '--warmup', '3', '--no-extra',
           '--no-e2e', '--no-cpu-baseline', '--no-torch-baseline', '--no-clocks', '--dump-outputs', str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    arrays = {f[:-len('.npy')]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}
    return arrays, json.loads(r.stdout)


def _sha(a, dtype):
    return hashlib.sha1(a.astype(dtype).tobytes()).hexdigest()[:16]


def test_dump_outputs_repeat_and_are_the_parity_round(tmp_path):
    cfg = synth.CONFIGS['C1']
    (a, line), (b, _) = _bench_dump(tmp_path / 'a'), _bench_dump(tmp_path / 'b')
    shapes = dict(labels=(cfg.n,), inertia=(1,), centers=(cfg.k, synth.D), topk_vals=(cfg.n, 5), topk_idx=(cfg.n, 5),
                  vote_names=(cfg.k, 20), vote_counts=(cfg.k, 20), vote_distinct=(cfg.k,), cluster_rows=(cfg.k,))
    assert {k: v.shape for k, v in a.items()} == shapes
    for k in shapes:
        assert a[k].dtype == (np.float32 if k in ('centers', 'topk_vals') else np.float64), k
        if k in ('centers', 'inertia'):
            assert np.allclose(a[k], b[k], rtol=1e-5, atol=1e-6), k
        else:
            assert np.array_equal(a[k], b[k]), k
    par = line['parity']
    assert _sha(a['labels'], np.int64) == par['labels_sha'] and _sha(a['topk_idx'], np.int64) == par['topk_idx_sha']
    assert _sha(a['vote_names'], np.int64) == par['voted_sha'] and _sha(a['vote_counts'], np.int32) == par['vote_counts_sha']
    assert np.array_equal(a['cluster_rows'], np.bincount(a['labels'].astype(np.int64), minlength=cfg.k))
