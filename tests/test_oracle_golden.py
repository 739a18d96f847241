"""The oracle is pinned here: every oracle function is compared with fixtures that were produced by
running the real reference code (oracle/gen_golden.py).  CPU only."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import hungarian_oracle, kmeans_oracle, naming_oracle

torch.set_num_threads(1)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_pairwise_distance_matches_reference(golden_dir):
    g = _load(golden_dir, 'kmeans_small.npz')
    X, C = torch.from_numpy(g['X']), torch.from_numpy(g['C0'])
    assert np.array_equal(kmeans_oracle.pairwise_distance(X, C, None).numpy(), g['pd_none'])
    assert np.array_equal(kmeans_oracle.pairwise_distance(X, C, 100).numpy(), g['pd_b100'])
    assert np.array_equal(kmeans_oracle.pairwise_distance(X, C, 600).numpy(), g['pd_b600'])
    assert kmeans_oracle.pairwise_distance(X[:0], C, 10).shape == (0, C.shape[0])


def test_blobs_demo_fit_mix(golden_dir):
    g = _load(golden_dir, 'kmeans_blobs_demo.npz')
    km = kmeans_oracle.K_Means(k=4, init='k-means++', random_state=1, n_jobs=None, pairwise_batch_size=10)
    km.fit_mix(torch.from_numpy(g['u_feats']), torch.from_numpy(g['l_feats']), torch.from_numpy(g['l_targets']))
    assert np.array_equal(km.labels_.numpy(), g['labels'])
    assert np.array_equal(km.cluster_centers_.numpy(), g['centers'])
    assert km.inertia_.item() == g['inertia']
    assert km.n_iter_ == g['n_iter'] == len(g['l_targets'])      # the reference's n_iter_ quirk


@pytest.mark.parametrize('tag,guard', [('local', False), ('gcd', True)])
def test_fit_mix_small(golden_dir, tag, guard):
    g = _load(golden_dir, 'kmeans_small.npz')
    km = kmeans_oracle.K_Means(k=12, tolerance=1e-4, max_iterations=10, init='k-means++', n_init=2,
                               random_state=7, n_jobs=None, pairwise_batch_size=128, mode=None,
                               guarded_kpp=guard)
    km.fit_mix(torch.from_numpy(g['u_feats']), torch.from_numpy(g['l_feats']), torch.from_numpy(g['l_targets']))
    assert np.array_equal(km.labels_.numpy(), g[f'mix_{tag}_labels'])
    assert np.array_equal(km.cluster_centers_.numpy(), g[f'mix_{tag}_centers'])
    assert km.inertia_.item() == g[f'mix_{tag}_inertia']
    assert km.n_iter_ == g[f'mix_{tag}_n_iter']


@pytest.mark.parametrize('init', ['random', 'first', 'k-means++'])
def test_fit_small(golden_dir, init):
    g = _load(golden_dir, 'kmeans_small.npz')
    tag = init.replace('-', '').replace('+', 'p')
    km = kmeans_oracle.K_Means(k=12, tolerance=1e-4, max_iterations=6, init=init, n_init=2,
                               random_state=3, n_jobs=None, pairwise_batch_size=None)
    km.fit(torch.from_numpy(g['X']))
    assert np.array_equal(km.labels_.numpy(), g[f'fit_{tag}_labels'])
    assert np.array_equal(km.cluster_centers_.numpy(), g[f'fit_{tag}_centers'])
    assert km.inertia_.item() == g[f'fit_{tag}_inertia']
    assert km.n_iter_ == g[f'fit_{tag}_n_iter']


def test_kpp_seeds(golden_dir):
    g = _load(golden_dir, 'kmeans_small.npz')
    X, u = torch.from_numpy(g['X']), torch.from_numpy(g['u_feats'])
    km = kmeans_oracle.K_Means(k=12, pairwise_batch_size=None)
    assert np.array_equal(km.kpp(X, k=12, random_state=5).numpy(), g['kpp_centers'])
    assert np.array_equal(km.kpp(u, pre_centers=X[:3].clone(), k=12, random_state=5).numpy(), g['kpp_pre_centers'])


def test_empty_cluster_gives_nan_row(golden_dir):
    g = _load(golden_dir, 'kmeans_empty_cluster.npz')
    km = kmeans_oracle.K_Means(k=5, max_iterations=1, init='first', n_init=1, random_state=0, pairwise_batch_size=None)
    km.fit(torch.from_numpy(g['X']))
    assert np.isnan(g['centers']).any(), 'fixture must contain the NaN row'
    assert np.array_equal(km.labels_.numpy(), g['labels'])
    assert np.array_equal(km.cluster_centers_.numpy(), g['centers'], equal_nan=True)


def test_hungarian_matches_reference(golden_dir):
    g = _load(golden_dir, 'hungarian.npz')
    n = 0
    for key in g.files:
        if key.startswith('cost_'):
            ind = hungarian_oracle.linear_assignment(g[key].copy())
            assert np.array_equal(ind, g['ind_' + key[5:]]), key
            n += 1
    assert n == 24


@pytest.mark.parametrize('n', [700, 2048, 2500])
def test_scoring_blocks(golden_dir, n):
    g = _load(golden_dir, 'naming_small.npz')
    feats, W = torch.from_numpy(g[f'feats_{n}']), torch.from_numpy(g['W'])
    idx, val = naming_oracle.score_topk(feats, W, 5, variant='unsup')
    assert np.array_equal(idx.numpy(), g[f'unsup_idx_{n}'])
    assert np.array_equal(val.numpy(), g[f'unsup_val_{n}'])
    idx, val = naming_oracle.score_topk(feats, W, 5, variant='ptsup')
    assert np.array_equal(idx.numpy(), g[f'ptsup_idx_{n}'])
    assert np.array_equal(val.numpy(), g[f'ptsup_val_{n}'])
    logits = 100. * feats[:512] @ W
    acc = naming_oracle.accuracy(logits, torch.from_numpy(g[f'acc_tgt_{n}']), topk=(1, 5))
    assert np.array_equal(np.array(acc), g[f'acc_{n}'])


def test_unsup_voting_loop(golden_dir):
    g = _load(golden_dir, 'naming_small.npz')
    n = 2500
    feats, W = torch.from_numpy(g[f'feats_{n}']), torch.from_numpy(g['W'])
    idx = torch.from_numpy(g[f'ptsup_idx_{n}'])
    trace = naming_oracle.naming_loop_unsup(idx, g['unsup_loop_preds0'].copy(), feats, W, n_cluster=10)
    assert len(trace) == int(g['unsup_loop_rounds']) >= 2
    for r, t in enumerate(trace):
        assert t['voted'] == g[f'unsup_loop_voted_{r}'].tolist()
        assert np.array_equal(t['u_preds'], g[f'unsup_loop_preds_{r}'])
        assert t['n_unique'] == int(g[f'unsup_loop_nuniq_{r}'])


def test_ptsup_voting_loop(golden_dir):
    g = _load(golden_dir, 'naming_small.npz')
    n = 2500
    feats, W = torch.from_numpy(g[f'feats_{n}']), torch.from_numpy(g['W'])
    idx = torch.from_numpy(g[f'ptsup_idx_{n}'])
    mask_lab = g['ptsup_loop_mask_lab']
    trace = naming_oracle.naming_loop_ptsup(idx[~mask_lab], g['ptsup_loop_all_preds'].copy(), mask_lab,
                                            feats[~mask_lab], W, g['ptsup_loop_lab_names'].tolist(), n_cluster=10)
    assert len(trace) == int(g['ptsup_loop_rounds']) >= 2
    for r, t in enumerate(trace):
        assert t['voted'] == g[f'ptsup_loop_voted_{r}'].tolist()
        assert t['cand'] == g[f'ptsup_loop_cand_{r}'].tolist()
        assert np.array_equal(t['u_preds'], g[f'ptsup_loop_preds_{r}'])


# ------------------------------------------------------------------ evaluation metrics (SURVEY 8f rank 4)
def _eval_cases(g):
    for ci in range(5):
        y, p, mask = g[f'c{ci}_y'], g[f'c{ci}_pred'], g[f'c{ci}_mask']
        names = {c: f'n{100 + c}' for c in range(int(g[f'c{ci}_ncls']))}
        yield ci, y, p, mask, names, [str(x) for x in g[f'c{ci}_cand']]


def test_split_cluster_acc_v2_reproduces_the_notebook_known_answer(golden_dir):
    """gcd/notebooks/demo_acc_v2.ipynb: 0.85 0.8 0.9 {2: 0, 1: 1, 0: 2, 3: 3} - the reference's one recorded answer"""
    from oracle import eval_oracle
    gt = np.array([0] * 5 + [1] * 5 + [2] * 5 + [3] * 5)
    pr = np.array([2] * 4 + [0] * 1 + [1] * 4 + [3] * 1 + [0] * 4 + [3] * 1 + [3] * 5)
    t, o, n, m = eval_oracle.split_cluster_acc_v2(gt, pr, gt < 2, return_ind_map=True)
    assert (t, o, n) == (0.85, 0.8, 0.9) and {int(k): int(v) for k, v in m.items()} == {2: 0, 1: 1, 0: 2, 3: 3}
    g = _load(golden_dir, 'eval_small.npz')
    assert np.array_equal(g['nb_acc'], [0.85, 0.8, 0.9])


def test_eval_oracle_matches_reference(golden_dir):
    from oracle import eval_oracle
    g = _load(golden_dir, 'eval_small.npz')
    for ci, y, p, mask, names, cand in _eval_cases(g):
        t, o, n, m = eval_oracle.split_cluster_acc_v2(y, p, mask, return_ind_map=True)
        assert np.array_equal(np.array([t, o, n]), g[f'c{ci}_acc'])                      # float64, bit-exact
        assert np.array_equal(np.array(sorted(m.items())), g[f'c{ci}_map'])
        for sub, sel in (('all', np.ones(len(y), bool)), ('old', mask), ('new', ~mask)):
            assert np.array_equal(np.array(eval_oracle.evaluate_semantic_acc(y[sel], names, p[sel], cand)), g[f'c{ci}_sem_{sub}'])


_PTSUP_STRINGS = """
import sys
from oracle import gen_golden as gg, naming_oracle
c = gg.ptsup_strings_case()
m = c['mask_lab']
got = naming_oracle.naming_loop_ptsup(c['idx_top'][~m], c['all_preds'].copy(), m, c['feats'][~m], c['W'], c['lab_idx'],
                                      c['k_true'], top_k=5, num_common_vote=20, num_common_linear=4, nouns=c['nouns'])
gg.save_ptsup_strings_trace(sys.argv[1], [(r['voted'], r['cand'], r['u_preds'], r['n_unique']) for r in got])
"""


def test_ptsup_loop_with_string_names_matches_the_stored_trace(golden_dir, tmp_path):
    """The partially supervised loop on a string vocabulary that is not in lexicographic order and holds duplicate names
    (``sorted(cand_names)`` sorts strings, ``nouns.index`` resolves duplicates to the first column), round by round
    against naming_ptsup_strings.npz.  The loop iterates string sets, so both run under the fixture's PYTHONHASHSEED."""
    from oracle import gen_golden as gg
    g = _load(golden_dir, 'naming_ptsup_strings.npz')
    assert str(g['hash_seed']) == gg.PTSUP_STRINGS_HASH_SEED
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONHASHSEED=gg.PTSUP_STRINGS_HASH_SEED)
    r = subprocess.run([sys.executable, '-c', _PTSUP_STRINGS, str(tmp_path / 'got.npz')], cwd=root, env=env,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(tmp_path / 'got.npz')
    assert int(got['rounds']) == int(g['rounds']) >= 2
    for k in g.files:
        assert got[k].dtype == g[k].dtype and np.array_equal(got[k], g[k]), k
    # the index-named shortcut would NOT have produced this: the lexicographic order differs from the column order
    nouns = gg.ptsup_strings_case()['nouns']
    cand = list(g['cand_0'])
    assert [nouns.index(s) for s in cand] != sorted(nouns.index(s) for s in cand)
