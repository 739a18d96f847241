#!/usr/bin/env python
"""Generate ``tests/golden/*.npz`` by running the REAL reference code on seeded inputs.

TEST INFRASTRUCTURE.  Runs only with a checkout of the reference project (not part of this repository);
the fixtures it writes are committed so that the tests never need the checkout.  Re-run with:
``PYTHONHASHSEED=0 python -m oracle.gen_golden --ref <checkout>`` (or SCD_REFERENCE_DIR=<checkout>).

``naming_ptsup_strings.npz`` was first written without a checkout, by ``oracle.naming_oracle.naming_loop_ptsup``, the
restatement that the live comparison in tests/test_golden_reproducible_cpu.py matched against the reference's loop
text; regenerating it from a checkout (``--only naming_strings``) replaces it with the reference's own trace, and that
test compares the two bit for bit.

What is executed from the reference (never copied into this repo):
  * imported as modules: ``local_utils/faster_mix_k_means_pytorch.py`` (K_Means, pairwise_distance),
    ``gcd/methods/clustering/faster_mix_k_means_pytorch.py`` (the copy the drivers import; ``mode=``),
    ``local_utils/clip_lang_util.py`` (assign_name, accuracy) and through it
    ``gcd/project_utils/cluster_utils.py`` (linear_assignment).  Import-time-only dependencies that
    are not installed (nltk, clip, matplotlib, seaborn, sklearn.utils._joblib) are stubbed.
  * exec'd from their source text, because they are inline script code under ``__main__``:
    ``main_unsup.py`` scoring block (TOP_K ... torch.cat) and voting loop (while ... argmax),
    ``main_ptsup.py`` scoring block and voting loop.  The line ranges are located by sentinel
    strings and the text is dedented and executed in a namespace holding the synthetic inputs.
"""
from __future__ import annotations

import argparse
import copy
import os
import sys
import textwrap
import types
from collections import Counter

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
OUT = os.path.join(REPO, 'tests', 'golden')


# ------------------------------------------------------------------ reference import plumbing
def _stub(name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    sys.modules[name] = mod
    return mod


def import_reference(ref):
    import joblib
    _stub('nltk')
    _stub('nltk.corpus', wordnet=None)
    _stub('clip')
    plt = _stub('matplotlib.pyplot', get=None)
    _stub('matplotlib', pyplot=plt, use=lambda *a, **k: None)
    _stub('seaborn')
    _stub('sklearn.utils._joblib', Parallel=joblib.Parallel, delayed=joblib.delayed,
          effective_n_jobs=joblib.effective_n_jobs)
    for p in (ref, os.path.join(ref, 'gcd'), os.path.join(ref, 'local_utils')):
        if p not in sys.path:
            sys.path.insert(0, p)
    import warnings
    warnings.simplefilter('ignore')
    import importlib
    km_local = importlib.import_module('local_utils.faster_mix_k_means_pytorch')
    km_gcd = importlib.import_module('gcd.methods.clustering.faster_mix_k_means_pytorch')
    lang = importlib.import_module('local_utils.clip_lang_util')
    cu = importlib.import_module('gcd.project_utils.cluster_utils')
    return km_local, km_gcd, lang, cu


def source_block(path, first_sentinel, last_sentinel, after=None):
    """Return the dedented text from the line containing ``first_sentinel`` (searched after the line
    containing ``after``, if given) through the line containing ``last_sentinel``, plus its 1-based range."""
    with open(path) as f:
        lines = f.readlines()
    start = 0
    if after is not None:
        start = next(i for i, l in enumerate(lines) if after in l) + 1
    a = next(i for i in range(start, len(lines)) if first_sentinel in lines[i])
    b = next(i for i in range(a, len(lines)) if last_sentinel in lines[i])
    return textwrap.dedent(''.join(lines[a:b + 1])), (a + 1, b + 1)


# ------------------------------------------------------------------ synthetic inputs
def unit_rows(x):
    return x / x.norm(dim=1, keepdim=True)


def clustered_feats(n, d, k_true, seed, spread=4.0):
    g = torch.Generator().manual_seed(seed)
    mu = unit_rows(torch.randn(k_true, d, generator=g))
    y = torch.randint(0, k_true, (n,), generator=g)
    x = unit_rows(torch.randn(n, d, generator=g) + spread * mu[y])
    return x.float().contiguous(), y


def bf16_round(x):
    return x.to(torch.bfloat16).to(torch.float32)


# ------------------------------------------------------------------ k-means fixtures
def gen_kmeans(km_local, km_gcd):
    from sklearn.datasets import make_blobs
    # (1) the reference's own demo, local_utils/faster_mix_k_means_pytorch.py:221-249 (float64 inputs!)
    X, y = make_blobs(n_samples=500, n_features=2, centers=4, cluster_std=1, center_box=(-10.0, 10.0),
                      shuffle=True, random_state=1)
    l_t, l_f, u_f = y[y > 1], X[y > 1], X[y < 2]
    km = km_local.K_Means(k=4, init='k-means++', random_state=1, n_jobs=None, pairwise_batch_size=10)
    km.fit_mix(torch.from_numpy(u_f), torch.from_numpy(l_f), torch.from_numpy(l_t))
    np.savez_compressed(os.path.join(OUT, 'kmeans_blobs_demo.npz'),
                        u_feats=u_f, l_feats=l_f, l_targets=l_t,
                        labels=km.labels_.numpy(), centers=km.cluster_centers_.numpy(),
                        inertia=np.float64(km.inertia_.item()), n_iter=np.int64(km.n_iter_))

    # (2) DINO-like unit-norm fp32 features, semi-supervised, both class copies, k-means++ and random
    n, d, k = 600, 64, 12
    X, y = clustered_feats(n, d, k, seed=11)
    lab = (y < k // 2) & (torch.rand(n, generator=torch.Generator().manual_seed(12)) < 0.5)
    l_f, u_f = X[lab].contiguous(), X[~lab].contiguous()
    l_t = y[lab].double()                                   # drivers pass float64 targets (main_unsup.py:118,132)
    C0 = X[:k].clone()
    out = dict(u_feats=u_f.numpy(), l_feats=l_f.numpy(), l_targets=l_t.numpy(), X=X.numpy(), C0=C0.numpy())
    out['pd_none'] = km_local.pairwise_distance(X, C0, None).numpy()
    out['pd_b100'] = km_local.pairwise_distance(X, C0, 100).numpy()
    out['pd_b600'] = km_local.pairwise_distance(X, C0, 600).numpy()
    for tag, mod, extra in (('local', km_local, {}), ('gcd', km_gcd, {'mode': None})):
        km = mod.K_Means(k=k, tolerance=1e-4, max_iterations=10, init='k-means++', n_init=2,
                         random_state=7, n_jobs=None, pairwise_batch_size=128, **extra)
        km.fit_mix(u_f, l_f, l_t)
        out[f'mix_{tag}_labels'] = km.labels_.numpy()
        out[f'mix_{tag}_centers'] = km.cluster_centers_.numpy()
        out[f'mix_{tag}_inertia'] = np.float64(km.inertia_.item())
        out[f'mix_{tag}_n_iter'] = np.int64(km.n_iter_)
    for init in ('random', 'first', 'k-means++'):
        km = km_local.K_Means(k=k, tolerance=1e-4, max_iterations=6, init=init, n_init=2,
                              random_state=3, n_jobs=None, pairwise_batch_size=None)
        km.fit(X)
        tag = init.replace('-', '').replace('+', 'p')
        out[f'fit_{tag}_labels'] = km.labels_.numpy()
        out[f'fit_{tag}_centers'] = km.cluster_centers_.numpy()
        out[f'fit_{tag}_inertia'] = np.float64(km.inertia_.item())
        out[f'fit_{tag}_n_iter'] = np.int64(km.n_iter_)
    # kpp seed selection alone (host RNG stream + cumsum threshold)
    km = km_local.K_Means(k=k, pairwise_batch_size=None)
    out['kpp_centers'] = km.kpp(X, k=k, random_state=5).numpy()
    out['kpp_pre_centers'] = km.kpp(u_f, pre_centers=X[:3].clone(), k=k, random_state=5).numpy()
    np.savez_compressed(os.path.join(OUT, 'kmeans_small.npz'), **out)

    # (3) empty cluster -> NaN centroid (duplicate first rows with the 'first k rows' init); one iteration
    Xd = X[:200].clone()
    Xd[1] = Xd[0]
    km = km_local.K_Means(k=5, max_iterations=1, init='first', n_init=1, random_state=0, pairwise_batch_size=None)
    km.fit(Xd)
    np.savez_compressed(os.path.join(OUT, 'kmeans_empty_cluster.npz'), X=Xd.numpy(),
                        labels=km.labels_.numpy(), centers=km.cluster_centers_.numpy(),
                        inertia=np.float64(km.inertia_.item()))


# ------------------------------------------------------------------ constrained k-means fixtures
def gen_constrained(ref):
    """Runs the REAL ``local_utils/sskm_constrained.py`` (graph construction, ``_labels_constrained``, ``fit`` /
    ``fit_mix``).  Its only missing dependency, the OR-Tools wrapper module
    ``k_means_constrained.mincostflow_vectorized`` (requirements.txt:103, not installed), is replaced by
    ``oracle.constrained_oracle.StandInMinCostFlow`` - so the solver is the stand-in, everything around it is the
    reference itself (parity unpinned for the solver, see the oracle's header)."""
    import importlib
    from oracle import constrained_oracle as co
    _stub('k_means_constrained')
    _stub('k_means_constrained.mincostflow_vectorized', SimpleMinCostFlowVectorized=co.StandInMinCostFlow)
    _stub('pyximport', install=lambda *a, **k: None)
    sk = importlib.import_module('local_utils.sskm_constrained')
    out = {}
    # (1) the 9 x 2 array of local_utils/test_kmeans_cons.py:3 with its parameters (k=2, size 2..5, random_state=0)
    X9 = torch.from_numpy(np.array([[1, 2], [1, 4], [1, 0], [4, 2], [4, 4], [4, 0], [4, 3], [4, 4], [4, 1]])).float()
    km = sk.K_Means(k=2, size_min=2, size_max=5, random_state=0)
    km.fit(X9)
    out['t9_X'] = X9.numpy()
    out['t9_labels'] = km.labels_.numpy()
    out['t9_centers'] = km.cluster_centers_.numpy()
    out['t9_inertia'] = np.float64(km.inertia_)
    out['t9_n_iter'] = np.int64(km.n_iter_)
    # (2) graph arrays + one constrained assignment on unit-norm features with ACTIVE bounds
    n, d, k = 240, 32, 6
    X, y = clustered_feats(n, d, k, seed=31)
    C0 = X[:k].clone()
    D_sqrt = torch.sqrt(sk.pairwise_distance(X, C0, None)).numpy()
    lo, hi = 36, 44
    edges, costs, caps, supplies, n_C, n_X = sk.minimum_cost_flow_problem_graph(X.numpy(), C0.numpy(), D_sqrt, lo, hi)
    labels, inertia = sk._labels_constrained(X.numpy(), C0.numpy(), D_sqrt, size_min=lo, size_max=hi,
                                             distances=np.zeros(n, dtype=np.float32))
    out.update(g_X=X.numpy(), g_C0=C0.numpy(), g_D_sqrt=D_sqrt, g_bounds=np.array([lo, hi]), g_edges=edges, g_costs=costs,
               g_caps=caps, g_supplies=supplies, g_labels=labels, g_inertia=np.float64(inertia),
               g_total_cost=np.int64(costs[:n * k].reshape(n, k)[np.arange(n), labels].sum()))
    # (3) whole fits: unsupervised (random init) and semi-supervised (k-means++ from the labelled means)
    km = sk.K_Means(k=k, tolerance=1e-4, max_iterations=5, size_min=lo, size_max=hi, init='random', n_init=2, random_state=4,
                    n_jobs=None, pairwise_batch_size=64)
    km.fit(X)
    out.update(fit_labels=km.labels_.numpy(), fit_centers=km.cluster_centers_.numpy(), fit_inertia=np.float64(km.inertia_),
               fit_n_iter=np.int64(km.n_iter_))
    lab = (y < k // 2) & (torch.rand(n, generator=torch.Generator().manual_seed(32)) < 0.5)
    l_f, u_f, l_t = X[lab].contiguous(), X[~lab].contiguous(), y[lab].double()
    lo_u, hi_u = 28, 36                               # bounds apply to the unlabelled rows only (:116)
    km = sk.K_Means(k=k, tolerance=1e-4, max_iterations=5, size_min=lo_u, size_max=hi_u, init='k-means++', n_init=2,
                    random_state=9, n_jobs=None, pairwise_batch_size=64)
    km.fit_mix(u_f, l_f, l_t)
    out.update(mix_u=u_f.numpy(), mix_l=l_f.numpy(), mix_t=l_t.numpy(), mix_bounds=np.array([lo_u, hi_u]),
               mix_labels=km.labels_.numpy(), mix_centers=km.cluster_centers_.numpy(),
               mix_inertia=np.float64(km.inertia_.item()), mix_n_iter=np.int64(km.n_iter_))
    np.savez_compressed(os.path.join(OUT, 'kmeans_constrained.npz'), **out)


# ------------------------------------------------------------------ Hungarian fixtures
def gen_hungarian(cu):
    rng = np.random.RandomState(0)
    out = {}
    shapes = [(1, 1), (2, 2), (3, 3), (5, 5), (8, 8), (13, 13), (20, 20), (33, 33), (40, 40), (4, 7), (7, 4), (12, 30)]
    for i, (r, c) in enumerate(shapes):
        for j, hi in enumerate((3, 50)):                  # hi=3 -> massively tied costs
            cost = rng.randint(0, hi, size=(r, c))
            out[f'cost_{i}_{j}'] = cost
            out[f'ind_{i}_{j}'] = cu.linear_assignment(cost.copy())
    np.savez_compressed(os.path.join(OUT, 'hungarian.npz'), **out)


# ------------------------------------------------------------------ naming fixtures
class _Args:
    pass


def gen_naming(ref, lang):
    d, v, k_true = 32, 300, 10
    res = {}
    unsup_src = os.path.join(ref, 'main_unsup.py')
    ptsup_src = os.path.join(ref, 'main_ptsup.py')

    score_unsup, r1 = source_block(unsup_src, 'TOP_K = args.topk', 'name_logits_top5 = torch.cat')
    score_ptsup, r2 = source_block(ptsup_src, 'TOP_K = 5', 'name_logits_top5 = torch.cat',
                                   after='## obtain top 5 predictions by CLIP')
    loop_unsup, r3 = source_block(unsup_src, 'while (set(cur_voted_names)', 'u_preds = logits.argmax')
    loop_ptsup, r4 = source_block(ptsup_src, 'while (set(cur_voted_names)', 'u_preds = logits.argmax')
    res['ranges'] = np.array([r1, r2, r3, r4])
    print('exec ranges: unsup score %s, ptsup score %s, unsup loop %s, ptsup loop %s' % (r1, r2, r3, r4))

    g = torch.Generator().manual_seed(21)
    W = bf16_round(unit_rows(torch.randn(v, d, generator=g))).t().contiguous()       # [D,V], V-contiguous
    res['W'] = W.numpy()
    for n in (700, 2048, 2500):              # < one batch, exact multiple (empty trailing batch), ragged
        feats, y = clustered_feats(n, d, k_true, seed=100 + n)
        feats = bf16_round(feats)
        args = _Args()
        args.topk = 5
        ns = dict(args=args, clip_all_feats=feats, zeroshot_weights=W, torch=torch, F=F, tqdm=lambda x: x)
        exec(score_unsup, ns)
        res[f'feats_{n}'] = feats.numpy()
        res[f'unsup_idx_{n}'] = ns['name_idx_top5'].numpy()
        res[f'unsup_val_{n}'] = ns['name_logits_top5'].numpy()
        ns = dict(clip_all_feats=feats, zeroshot_weights=W, torch=torch, F=F, tqdm=lambda x: x)
        exec(score_ptsup, ns)
        res[f'ptsup_idx_{n}'] = ns['name_idx_top5'].numpy()
        res[f'ptsup_val_{n}'] = ns['name_logits_top5'].numpy()
        # accuracy() on full logits of the first 512 rows against synthetic targets
        logits = 100. * feats[:512] @ W
        tgt = torch.randint(0, v, (512,), generator=torch.Generator().manual_seed(n))
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            res[f'acc_{n}'] = np.array(lang.accuracy(logits, tgt, topk=(1, 5)))
        res[f'acc_tgt_{n}'] = tgt.numpy()

    # ---- voting loops on n = 2500 (names are ints: nouns[i] == i, so set/sort order is hash-seed free)
    n = 2500
    feats = torch.from_numpy(res[f'feats_{n}'])
    idx_top = torch.from_numpy(res[f'ptsup_idx_{n}'])
    _, y = clustered_feats(n, d, k_true, seed=100 + n)
    g2 = torch.Generator().manual_seed(5)
    noise = torch.randint(0, k_true, (n,), generator=g2)
    flip = torch.rand(n, generator=g2) < 0.15
    preds0 = torch.where(flip, noise, y).numpy().astype(np.int64)        # imperfect clustering result
    nouns = list(range(v))
    rec = []

    def fake_split_acc(y_true, y_pred, mask, return_ind_map=False):
        rec.append(np.array(y_pred).copy())
        return (0., 0., 0., {}) if return_ind_map else (0., 0., 0.)

    args = _Args()
    args.num_common_vote, args.num_common_linear, args.n_cluster, args.dataset_name = 20, 4, k_true, 'cub'
    voted = []

    def fake_sem_acc(t, c2n, p, cand_names):
        if not voted or voted[-1] is not cand_names:
            voted.append(cand_names)
        return 0., 0.

    ns = dict(args=args, name_idx_top5=idx_top, u_preds=preds0.copy(), nouns=nouns, zeroshot_weights=W,
              clip_u_feats=feats, num_unlab_classes=k_true, cur_voted_names=[0.5], prev_voted_names=[1.5],
              top_k=5, it=0, Counter=Counter, copy=copy, torch=torch, assign_name=lang.assign_name,
              split_cluster_acc_v2=fake_split_acc, evaluate_semantic_acc=fake_sem_acc,
              u_targets=None, mask=None, cidx_to_cname=None, print=lambda *a, **k: None)
    # the exec'd text ends at the argmax line; the metric calls after it are outside the block, so
    # run the block round by round: it is a ``while`` loop -> wrap to record each round.
    loop_body_unsup = loop_unsup.replace('u_preds = logits.argmax(dim=-1).view(-1).cpu().numpy()',
                                         'u_preds = logits.argmax(dim=-1).view(-1).cpu().numpy()\n'
                                         '    _rec(cur_voted_names, u_preds, len(voted_unique_name_idx))')
    trace = []
    ns['_rec'] = lambda names, p, nu: trace.append((list(names), np.array(p).copy(), nu))
    exec(loop_body_unsup, ns)
    res['unsup_loop_preds0'] = preds0
    res['unsup_loop_rounds'] = np.int64(len(trace))
    for r, (names, p, nu) in enumerate(trace):
        res[f'unsup_loop_voted_{r}'] = np.array(names, dtype=np.int64)
        res[f'unsup_loop_preds_{r}'] = p.astype(np.int64)
        res[f'unsup_loop_nuniq_{r}'] = np.int64(nu)

    # ptsup: first k_true//2 classes are labelled; labelled rows get their class as cluster id
    mask_lab = ((y < k_true // 2) & (torch.rand(n, generator=torch.Generator().manual_seed(6)) < 0.5)).numpy()
    all_preds = preds0.copy()
    all_preds[mask_lab] = y.numpy()[mask_lab]
    lab_names = [int(idx_top[(y == c).numpy() & mask_lab][:, 0].mode().values) for c in range(k_true // 2)]
    lab_names = list(dict.fromkeys(lab_names))                 # distinct, order kept
    u_preds = all_preds[~mask_lab]
    l_preds = all_preds[mask_lab]
    trace = []
    ns = dict(args=args, name_idx_top5=idx_top[~mask_lab], u_preds=u_preds.copy(), nouns=nouns,
              zeroshot_weights=W, clip_u_feats=feats[~mask_lab], lab_names=lab_names,
              num_unlab_classes=k_true - len(lab_names), known_name_idx=[nouns.index(x) for x in lab_names],
              unlab_cluster_idx=list(set(list(set(all_preds))) - set(list(set(l_preds)))),
              cur_voted_names=[0.5], prev_voted_names=[1.5], top_k=5, it=0, Counter=Counter, copy=copy,
              torch=torch, assign_name=lang.assign_name, print=lambda *a, **k: None,
              _rec=lambda names, cand, p, nu: trace.append((list(names), list(cand), np.array(p).copy(), nu)))
    loop_body_ptsup = loop_ptsup.replace('u_preds = logits.argmax(dim=-1).view(-1).cpu().numpy()',
                                         'u_preds = logits.argmax(dim=-1).view(-1).cpu().numpy()\n'
                                         '    _rec(cur_voted_names, cand_names, u_preds, len(voted_unique_name_idx))')
    exec(loop_body_ptsup, ns)
    res['ptsup_loop_all_preds'] = all_preds
    res['ptsup_loop_mask_lab'] = mask_lab
    res['ptsup_loop_lab_names'] = np.array(lab_names, dtype=np.int64)
    res['ptsup_loop_rounds'] = np.int64(len(trace))
    for r, (names, cand, p, nu) in enumerate(trace):
        res[f'ptsup_loop_voted_{r}'] = np.array(names, dtype=np.int64)
        res[f'ptsup_loop_cand_{r}'] = np.array(cand, dtype=np.int64)
        res[f'ptsup_loop_preds_{r}'] = p.astype(np.int64)
        res[f'ptsup_loop_nuniq_{r}'] = np.int64(nu)
    np.savez_compressed(os.path.join(OUT, 'naming_small.npz'), **res)


PTSUP_STRINGS_HASH_SEED = '0'


def ptsup_strings_case():
    """Inputs of the partially supervised voting loop with STRING names: the vocabulary is not in lexicographic order and
    holds duplicate names (``sorted(cand_names)`` main_ptsup.py:659 sorts strings, ``nouns.index`` resolves a duplicate to
    its first column).  The loop's ``list(set(...) - set(...))`` order depends on string hashing, so a trace of it is only
    reproducible under a fixed PYTHONHASHSEED (PTSUP_STRINGS_HASH_SEED)."""
    d, v, k_true, n = 32, 300, 10, 2500
    g = torch.Generator().manual_seed(21)
    W = bf16_round(unit_rows(torch.randn(v, d, generator=g))).t().contiguous()
    feats, y = clustered_feats(n, d, k_true, seed=100 + n)
    feats = bf16_round(feats)
    idx_top = (100. * feats @ W).topk(5, 1, True, True)[1]
    rs = np.random.RandomState(3)
    nouns = ['n%05d' % x for x in rs.permutation(v)]                  # column order != lexicographic order
    for a, b in ((7, 150), (20, 21), (40, 299)):                      # duplicate names: nouns.index -> first column
        nouns[b] = nouns[a]
    g2 = torch.Generator().manual_seed(5)
    noise = torch.randint(0, k_true, (n,), generator=g2)
    flip = torch.rand(n, generator=g2) < 0.15
    preds0 = torch.where(flip, noise, y).numpy().astype(np.int64)
    mask_lab = ((y < k_true // 2) & (torch.rand(n, generator=torch.Generator().manual_seed(6)) < 0.5)).numpy()
    all_preds = preds0.copy()
    all_preds[mask_lab] = y.numpy()[mask_lab]
    lab_idx = [int(idx_top[(y == c).numpy() & mask_lab][:, 0].mode().values) for c in range(k_true // 2)]
    lab_idx = list(dict.fromkeys(lab_idx))
    lab_names = list(dict.fromkeys(nouns[i] for i in lab_idx))
    lab_idx = [nouns.index(s) for s in lab_names]
    return dict(W=W, feats=feats, idx_top=idx_top, nouns=nouns, all_preds=all_preds, mask_lab=mask_lab, lab_idx=lab_idx,
                lab_names=lab_names, k_true=k_true)


def run_reference_ptsup_strings(ref, lang, c):
    """The reference's own loop text (main_ptsup.py) on ``ptsup_strings_case()``: per round (voted names, candidate
    names, u_preds, number of distinct voted names)."""
    loop_ptsup, _ = source_block(os.path.join(ref, 'main_ptsup.py'), 'while (set(cur_voted_names)', 'u_preds = logits.argmax')
    mask_lab, all_preds, nouns, k_true = c['mask_lab'], c['all_preds'], c['nouns'], c['k_true']
    u_preds, l_preds = all_preds[~mask_lab], all_preds[mask_lab]
    args = _Args()
    args.num_common_vote, args.num_common_linear, args.n_cluster, args.dataset_name = 20, 4, k_true, 'cub'
    trace = []
    ns = dict(args=args, name_idx_top5=c['idx_top'][~mask_lab], u_preds=u_preds.copy(), nouns=nouns,
              zeroshot_weights=c['W'], clip_u_feats=c['feats'][~mask_lab], lab_names=c['lab_names'],
              num_unlab_classes=k_true - len(c['lab_names']), known_name_idx=[nouns.index(x) for x in c['lab_names']],
              unlab_cluster_idx=list(set(list(set(all_preds))) - set(list(set(l_preds)))),
              cur_voted_names=[0.5], prev_voted_names=[1.5], top_k=5, it=0, Counter=Counter, copy=copy,
              torch=torch, assign_name=lang.assign_name, print=lambda *a, **k: None,
              _rec=lambda names, cand, p, nu: trace.append((list(names), list(cand), np.array(p).copy(), nu)))
    body = loop_ptsup.replace('u_preds = logits.argmax(dim=-1).view(-1).cpu().numpy()',
                              'u_preds = logits.argmax(dim=-1).view(-1).cpu().numpy()\n'
                              '    _rec(cur_voted_names, cand_names, u_preds, len(voted_unique_name_idx))')
    exec(body, ns)
    return trace


def save_ptsup_strings_trace(path, trace):
    out = dict(rounds=np.int64(len(trace)), hash_seed=np.array(PTSUP_STRINGS_HASH_SEED))
    for r, (names, cand, p, nu) in enumerate(trace):
        out.update({f'voted_{r}': np.array(names, dtype=str), f'cand_{r}': np.array(cand, dtype=str),
                    f'preds_{r}': np.asarray(p, dtype=np.int64), f'nuniq_{r}': np.int64(nu)})
    np.savez_compressed(path, **out)


def gen_naming_strings(ref, lang):
    if os.environ.get('PYTHONHASHSEED') != PTSUP_STRINGS_HASH_SEED:
        raise SystemExit(f'naming_strings: run with PYTHONHASHSEED={PTSUP_STRINGS_HASH_SEED} (the loop iterates string sets)')
    save_ptsup_strings_trace(os.path.join(OUT, 'naming_ptsup_strings.npz'),
                             run_reference_ptsup_strings(ref, lang, ptsup_strings_case()))


# ------------------------------------------------------------------ evaluation + on-disk contract fixtures
class _FakeImages:
    """Stands in for an image batch: ``extract_feature`` only calls ``.cuda()`` on it and hands it to the model."""

    def __init__(self, feats):
        self.feats = feats

    def cuda(self):
        return self


def gen_eval(ref):
    """Runs the REAL ``split_cluster_acc_v2`` (imported), ``evaluate_semantic_acc`` and ``extract_feature`` (exec'd from
    the source text of ``main_unsup.py``: the module itself does not import without matplotlib) on seeded inputs, and
    writes the dicts the drivers ``torch.save`` (``main_unsup.py:294-300`` features, ``:366-371`` cluster result)."""
    import importlib
    from collections import defaultdict
    clu = importlib.import_module('gcd.project_utils.cluster_and_log_utils')
    unsup_src = os.path.join(ref, 'main_unsup.py')
    sem_src, r1 = source_block(unsup_src, 'def evaluate_semantic_acc', 'return semantic_acc_avg, semantic_acc_all')
    ext_src, r2 = source_block(unsup_src, 'def extract_feature', 'return data_dict')
    ns = dict(defaultdict=defaultdict, np=np, torch=torch, tqdm=lambda x: x, print=lambda *a, **k: None)
    exec(sem_src, ns)
    exec(ext_src, ns)
    res = dict(ranges=np.array([r1, r2]))
    # (1) the reference's own known-answer case, gcd/notebooks/demo_acc_v2.ipynb
    gt = np.array([0] * 5 + [1] * 5 + [2] * 5 + [3] * 5)
    pr = np.array([2] * 4 + [0] * 1 + [1] * 4 + [3] * 1 + [0] * 4 + [3] * 1 + [3] * 5)
    t, o, n_, m = clu.split_cluster_acc_v2(gt, pr, gt < 2, return_ind_map=True)
    assert (t, o, n_, m) == (0.85, 0.8, 0.9, {2: 0, 1: 1, 0: 2, 3: 3}), (t, o, n_, m)
    res.update(nb_gt=gt, nb_pred=pr, nb_acc=np.array([t, o, n_]), nb_map=np.array(sorted(m.items())))
    # (2) seeded cases: float64 targets as the drivers pass them, more clusters than classes and vice versa, ties
    rng = np.random.RandomState(41)
    cases = [(400, 7, 7, 0.2), (1500, 12, 9, 0.35), (1500, 9, 14, 0.35), (64, 5, 5, 0.9), (3000, 40, 40, 0.1)]
    for ci, (n, n_cls, n_clu, noise) in enumerate(cases):
        y = rng.randint(0, n_cls, size=n)
        perm = rng.permutation(max(n_cls, n_clu))
        pred = np.where(rng.rand(n) < noise, rng.randint(0, n_clu, size=n), perm[y] % n_clu).astype(np.int64)
        mask = y < n_cls // 2
        y_f = y.astype(np.float64)
        t, o, n_, m = clu.split_cluster_acc_v2(y_f, pred, mask, return_ind_map=True)
        res[f'c{ci}_y'] = y_f
        res[f'c{ci}_pred'] = pred
        res[f'c{ci}_mask'] = mask
        res[f'c{ci}_acc'] = np.array([t, o, n_], dtype=np.float64)
        res[f'c{ci}_map'] = np.array(sorted(m.items()), dtype=np.int64)
        # semantic accuracy: class c is called name 100 + c; cluster p was voted name 100 + (class it mostly holds),
        # two clusters share a name and one name is unknown to every cluster
        cidx_to_cname = {c: f'n{100 + c}' for c in range(n_cls)}
        D = max(n_cls, n_clu)
        w = np.zeros((D, D), dtype=int)
        np.add.at(w, (pred, y), 1)
        cand = [f'n{100 + int(w[p].argmax())}' for p in range(n_clu)]
        cand[-1] = 'n_none'
        for sub, sel in (('all', np.ones(n, bool)), ('old', mask), ('new', ~mask)):
            a, b = ns['evaluate_semantic_acc'](y_f[sel], cidx_to_cname, pred[sel], cand)
            res[f'c{ci}_sem_{sub}'] = np.array([a, b], dtype=np.float64)
        res[f'c{ci}_cand'] = np.array(cand)
        res[f'c{ci}_ncls'] = np.int64(n_cls)
    np.savez_compressed(os.path.join(OUT, 'eval_small.npz'), **res)

    # (3) on-disk contracts: the dict extract_feature returns (main_unsup.py:113-146) saved as the drivers do
    # (:298), and the cluster-result dict (:366-371)
    g = torch.Generator().manual_seed(51)
    n, d = 300, 16
    raw = torch.randn(n, d, generator=g)
    labels = torch.randint(0, 8, (n,), generator=g)
    lab_mask = (labels < 4) & (torch.rand(n, generator=g) < 0.5)
    loader = [(_FakeImages(raw[i:i + 128]), labels[i:i + 128], None, lab_mask[i:i + 128]) for i in range(0, n, 128)]
    args = _Args()
    args.train_classes, args.feat_model = range(4), 'dino'
    data_dict = ns['extract_feature'](lambda im: im.feats, loader, args)
    torch.save(data_dict, os.path.join(OUT, 'features_all.pt'))
    mask_lab = data_dict['mask_lab']
    all_preds = rng.randint(0, 8, size=n)
    cluster_result = {'all_preds': all_preds}
    cluster_result['u_preds'] = all_preds[~mask_lab]
    cluster_result['u_targets'] = data_dict['targets'][~mask_lab]
    cluster_result['mask'] = data_dict['mask_cls'][~mask_lab].astype(bool)
    torch.save(cluster_result, os.path.join(OUT, 'cluster_result.pt'))
    np.savez_compressed(os.path.join(OUT, 'features_raw.npz'), raw=raw.numpy(), labels=labels.numpy(), lab_mask=lab_mask.numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ref', default=os.environ.get('SCD_REFERENCE_DIR'), help='checkout of the reference project')
    ap.add_argument('--out', default=None, help='write the fixtures here instead of tests/golden (used by the reproducibility test)')
    ap.add_argument('--only', default=None, choices=[None, 'kmeans', 'constrained', 'hungarian', 'naming', 'naming_strings', 'eval'],
                    help='regenerate one fixture family (the others are left as committed)')
    a = ap.parse_args()
    if not a.ref:
        ap.error('--ref (or SCD_REFERENCE_DIR) must name a checkout of the reference project')
    global OUT
    if a.out:
        OUT = os.path.abspath(a.out)
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)          # fixtures must not depend on the thread count of this box
    km_local, km_gcd, lang, cu = import_reference(a.ref)
    todo = lambda name: a.only in (None, name)
    if todo('kmeans'):
        gen_kmeans(km_local, km_gcd)
    if todo('constrained'):
        gen_constrained(a.ref)
    if todo('hungarian'):
        gen_hungarian(cu)
    if todo('naming'):
        gen_naming(a.ref, lang)
    if todo('naming_strings'):
        gen_naming_strings(a.ref, lang)
    if todo('eval'):
        gen_eval(a.ref)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == '__main__':
    main()
