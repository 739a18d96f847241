"""CPU-only: the C-ABI library builds, loads and exports every symbol include/scd_b200.h declares; the
host-side pieces that need no GPU (Munkres, workspace sizing) behave."""
import ctypes
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    with open(os.path.join(ROOT, 'include', 'scd_b200.h')) as f:
        text = f.read()
    return sorted(set(re.findall(r'SCD_API\s+[\w\s\*]+?\b(scd_\w+)\s*\(', text)))


def test_header_declares_the_expected_surface():
    syms = _declared_symbols()
    for must in ('scd_estep', 'scd_mstep_sums', 'scd_finalize_centers', 'scd_pairwise_distance', 'scd_name_topk',
                 'scd_topk_merge', 'scd_vote', 'scd_vocab_prepare', 'scd_linear_assignment', 'scd_last_error'):
        assert must in syms


def test_library_builds_and_exports_every_declared_symbol():
    from scd_b200 import _lib, build
    path = build.build()
    assert os.path.exists(path)
    lib = _lib.load()
    declared = _declared_symbols()
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in scd_b200.h but not exported'
    assert sorted(_lib.SIGNATURES) == declared, 'ctypes signatures out of sync with the header'
    assert lib.scd_version() == 200


def test_workspace_sizes_are_sane_without_a_gpu():
    from scd_b200 import _lib
    lib = _lib.load()
    assert lib.scd_mstep_workspace_bytes(1000, 10) >= (1000 + 21) * 4
    assert lib.scd_vote_workspace_bytes(1000, 10) >= (1000 + 31) * 4
    small = lib.scd_name_topk_workspace_bytes(1000, 3000, 5)
    big = lib.scd_name_topk_workspace_bytes(127000, 21000, 5)
    assert 1000 * 5 * 8 <= small and 127000 * 5 * 8 <= big < 127000 * 5 * 8 * 20


def test_removed_one_pass_em_is_refused_without_device_work():
    """assign_from_host keeps its mstep= keyword but refuses a value before touching the device, and the E-step
    reports no one-pass E+M plan (called unbound: constructing an _EStep allocates on the device)."""
    import pytest
    import torch
    from scd_b200 import kmeans
    with pytest.raises(ValueError, match='one-pass E\\+M was removed'):
        kmeans.assign_from_host(np.zeros((4, 8), np.float32), torch.zeros(2, 8), mstep=object())
    assert kmeans._EStep.fusable(object(), 127000) is False


def test_munkres_tie_breaking_matches_reference(golden_dir):
    from scd_b200 import naming
    g = np.load(os.path.join(golden_dir, 'hungarian.npz'))
    n = 0
    for key in g.files:
        if key.startswith('cost_'):
            assert np.array_equal(naming.linear_assignment(g[key]), g['ind_' + key[5:]]), key
            n += 1
    assert n == 24
    assert naming.linear_assignment(np.zeros((0, 0))).shape == (0, 2)


def test_assign_name_matches_oracle():
    from collections import Counter
    from oracle import naming_oracle
    from scd_b200 import naming
    rng = np.random.RandomState(1)
    c2c = {c: Counter({np.int64(n): int(v) for n, v in zip(rng.choice(60, 12, replace=False), rng.randint(1, 6, 12))})
           for c in range(9)}
    uniq = list(set(n for c in c2c for n, _ in c2c[c].most_common(20)))
    ind_o, w_o = naming_oracle.assign_name(uniq, c2c, num_common=4)
    ind, w = naming.assign_name(uniq, c2c, num_common=4)
    assert np.array_equal(w, w_o) and np.array_equal(ind, ind_o)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'scd_b200')
    for fn in os.listdir(pkg):
        if fn.endswith('.py'):
            with open(os.path.join(pkg, fn)) as f:
                src = f.read()
            assert not re.search(r'^\s*(from|import)\s+oracle\b', src, flags=re.M), fn
