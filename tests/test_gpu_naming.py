"""GPU parity: fused scoring/top-k, vote, assign/re-assign loops through the C ABI against the oracle and
the reference-generated golden fixtures.

Tolerances (BASELINE.json north_star): scores within 1e-4 absolute on the cosine scale, i.e. 1e-2 on the
x100 logits (asserted tighter: 2e-3); softmax probabilities within 1e-5; top-k indices bit-exact wherever
the gap to the neighbouring score exceeds TAU = 1e-3 logits (1e-5 cosine)."""
import os

import numpy as np
import pytest
import torch

from oracle import naming_oracle
from scd_b200 import kmeans, naming, synth

pytestmark = pytest.mark.gpu
TAU = 1e-3
LOGIT_ATOL = 2e-3


def _oracle_topk(feats, W, k, variant):
    """oracle top-(k+1) so the k-th/(k+1)-th gap is known"""
    kk = min(k + 1, W.shape[1])
    idx, val = naming_oracle.score_topk(feats, W, kk, variant=variant)
    return idx, val


def _check_topk(vals, idx, feats, W, k, variant, atol):
    """values within atol of the oracle; indices equal wherever the logit gaps to both neighbours (including
    the (k+1)-th score) exceed TAU"""
    oi, ov = _oracle_topk(feats, W, k, variant)
    kk = min(k, W.shape[1])
    vals, idx = vals.cpu()[:, :kk], idx.cpu()[:, :kk]
    assert torch.allclose(vals, ov[:, :kk], atol=atol, rtol=0), float((vals - ov[:, :kk]).abs().max())
    # margins are defined on the logits (the softmax is monotone, its probabilities are not on that scale)
    lv = ov if variant == 'ptsup' else _oracle_topk(feats, W, k, 'ptsup')[1]
    n = len(feats)
    gaps = lv[:, :-1] - lv[:, 1:] if lv.shape[1] > 1 else torch.full((n, 0), 1e9)
    if lv.shape[1] == kk:                       # no (k+1)-th score (k >= V): the last entry has no right neighbour
        gaps = torch.cat((gaps, torch.full((n, 1), 1e9)), dim=1)
    clear = gaps > TAU                          # [n, kk]: gap between entry j and entry j+1
    left = torch.cat((torch.ones(n, 1, dtype=torch.bool), clear[:, :kk - 1]), dim=1)
    pinned = left & clear[:, :kk]
    assert pinned.float().mean() > 0.97
    assert torch.equal(idx[pinned], oi[:, :kk][pinned])
    return pinned.float().mean().item()


@pytest.mark.parametrize('n', [700, 2048, 2500])
def test_scoring_matches_reference_golden(golden_dir, n):
    g = np.load(os.path.join(golden_dir, 'naming_small.npz'))
    feats, W = torch.from_numpy(g[f'feats_{n}']), torch.from_numpy(g['W'])
    vals, idx = naming.score_topk(feats, W, k=5, softmax=False)
    assert idx.dtype == torch.int64 and idx.shape == (n, 5) and vals.is_cuda
    assert np.allclose(vals.cpu().numpy(), g[f'ptsup_val_{n}'], atol=LOGIT_ATOL, rtol=0)
    _check_topk(vals, idx, feats, W, 5, 'ptsup', LOGIT_ATOL)
    vals, idx = naming.score_topk(feats, W, k=5, softmax=True)
    assert np.allclose(vals.cpu().numpy(), g[f'unsup_val_{n}'], atol=1e-5, rtol=1e-4)
    _check_topk(vals, idx, feats, W, 5, 'unsup', 1e-5)
    tgt = torch.from_numpy(g[f'acc_tgt_{n}'])
    assert naming.accuracy(feats[:512], W, tgt, topk=(1, 5)) == g[f'acc_{n}'].tolist()


@pytest.mark.parametrize('n,v,d,k', [(1, 1, 64, 1), (513, 257, 72, 2), (100, 255, 768, 3), (300, 256, 64, 5),
                                     (300, 5000, 768, 5), (1000, 3000, 768, 8), (2500, 1000, 512, 1), (4000, 21000, 768, 5)])
def test_scoring_shapes_against_oracle(n, v, d, k):
    g = torch.Generator().manual_seed(n + v + d + k)
    feats = synth.bf16_round(synth.unit_rows(torch.randn(n, d, generator=g)))
    W = synth.vocabulary(v, seed=n + v, d=d)
    vals, idx = naming.score_topk(feats, W, k=k, softmax=False)
    _check_topk(vals, idx, feats, W, k, 'ptsup', LOGIT_ATOL)
    if k > v:
        assert (idx.cpu()[:, v:] == -1).all()
    assert torch.equal(naming.clip_preds(feats, W).cpu(), idx.cpu()[:, 0])


def test_ndarray_features_and_prepared_vocabulary():
    g = torch.Generator().manual_seed(4)
    feats = synth.bf16_round(synth.unit_rows(torch.randn(900, 128, generator=g)))
    W = synth.vocabulary(700, seed=4, d=128)
    vocab = naming.Vocabulary(W.cuda())
    v1, i1 = naming.score_topk(feats.numpy(), vocab, k=5)           # ndarray in, like main_unsup.py:522
    v2, i2 = naming.score_topk(feats.cuda(), W.cuda().bfloat16(), k=5)
    assert torch.equal(i1, i2) and torch.equal(v1, v2)


def test_vocabulary_shards_merge_to_the_unsharded_result():
    """Column-sharded vocabulary (SURVEY 8e): local top-k per shard with global indices + k-way merge equals
    the single-shard answer; softmax needs the per-shard (max, sum-exp)."""
    from scd_b200 import dist as sdist
    g = torch.Generator().manual_seed(8)
    feats = synth.bf16_round(synth.unit_rows(torch.randn(1500, 768, generator=g)))
    W = synth.vocabulary(4099, seed=8)
    fb = naming._feats_bf16(feats)
    for softmax in (False, True):
        want_v, want_i = naming.score_topk(feats, W, k=5, softmax=softmax)
        parts = []
        for r in range(3):
            lo, hi = sdist.shard_bounds(4099, 3, r)
            vocab = naming.Vocabulary(W[:, lo:hi].cuda(), col_offset=lo)
            parts.append(naming.name_topk_raw(fb, vocab, 5, False, want_stats=True))
        got_v, got_i = sdist.merge_topk_parts(parts, 5, softmax)
        assert torch.equal(got_i, want_i)
        assert torch.allclose(got_v, want_v, atol=1e-6 if softmax else 1e-5, rtol=1e-5)


def _counter_list(c, m=20):
    return [(int(a), int(b)) for a, b in c.most_common(m)]


@pytest.mark.parametrize('known', [None, [1, 2, 3, 7]])
def test_vote_matches_oracle_counters(known):
    g = torch.Generator().manual_seed(3)
    n, k, v = 20000, 37, 900
    idx = torch.randint(0, v, (n, 5), generator=g)
    idx[:, 0] = torch.randint(0, 40, (n,), generator=g)             # many ties in the counts
    preds = torch.randint(0, k, (n,), generator=g).numpy()
    preds[preds == 5] = 6                                            # cluster 5 is empty
    for top_k in (5, 2):
        co = naming_oracle.vote(idx, preds, list(range(k)), top_k, known_name_idx=known)
        cg = naming.vote(idx.cuda(), preds, list(range(k)), top_k, 20, known_name_idx=known)
        for c in range(k):
            assert _counter_list(cg[c]) == _counter_list(co[c]), c
        assert naming.voted_candidates(cg, list(range(k)), 20) == naming_oracle.voted_candidates(co, list(range(k)), 20)
    names, counts, distinct, rows, ovf = naming.vote_device(idx.cuda(), preds, k, 5, 20, known)
    assert int(ovf) == 0 and torch.equal(rows.cpu().long(), torch.bincount(torch.from_numpy(preds), minlength=k))
    assert [int(x) for x in distinct.cpu()] == [len(co_c) for co_c in naming_oracle.vote(idx, preds, list(range(k)), 5, known_name_idx=known).values()]
    # the same vote on the label sort the M-step has just made (scd_vote_presorted): that sort is not stable, the vote's
    # first-occurrence tie order must not depend on it
    ms = kmeans._MStep(n, 4, k, 'cuda')
    ms.sums_counts(torch.randn(n, 4, generator=torch.Generator().manual_seed(4)).cuda(), torch.from_numpy(preds).cuda())
    for top_k in (5, 2):
        co = naming_oracle.vote(idx, preds, list(range(k)), top_k, known_name_idx=known)
        names, counts, distinct, rows, ovf = naming.vote_device(idx.cuda(), None, k, top_k, 20, known, presorted=ms)
        assert int(ovf) == 0 and torch.equal(rows.cpu().long(), torch.bincount(torch.from_numpy(preds), minlength=k))
        for c in range(k):
            assert [(int(a), int(b)) for a, b in zip(names[c].tolist(), counts[c].tolist()) if a >= 0] == _counter_list(co[c]), c
            assert int(distinct[c]) == len(co[c])


def test_unsup_voting_loop_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'naming_small.npz'))
    n = 2500
    feats, W = torch.from_numpy(g[f'feats_{n}']), torch.from_numpy(g['W'])
    _, idx = naming.score_topk(feats, W, k=5)
    trace = naming.naming_loop_unsup(idx, g['unsup_loop_preds0'].copy(), feats, W, n_cluster=10)
    assert len(trace) == int(g['unsup_loop_rounds'])
    for r, t in enumerate(trace):
        assert t['voted'] == g[f'unsup_loop_voted_{r}'].tolist()
        assert t['n_unique'] == int(g[f'unsup_loop_nuniq_{r}'])
        assert (t['u_preds'] == g[f'unsup_loop_preds_{r}']).mean() > 0.999


def test_ptsup_voting_loop_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'naming_small.npz'))
    n = 2500
    feats, W = torch.from_numpy(g[f'feats_{n}']), torch.from_numpy(g['W'])
    mask_lab = g['ptsup_loop_mask_lab']
    _, idx = naming.score_topk(feats, W, k=5)
    trace = naming.naming_loop_ptsup(idx[torch.from_numpy(~mask_lab).cuda()], g['ptsup_loop_all_preds'].copy(), mask_lab,
                                     feats[~mask_lab], W, g['ptsup_loop_lab_names'].tolist(), n_cluster=10)
    assert len(trace) == int(g['ptsup_loop_rounds'])
    for r, t in enumerate(trace):
        assert t['voted'] == g[f'ptsup_loop_voted_{r}'].tolist()
        assert t['cand'] == g[f'ptsup_loop_cand_{r}'].tolist()
        assert (t['u_preds'] == g[f'ptsup_loop_preds_{r}']).mean() > 0.999


def test_full_size_c2_properties():
    """127k x 768 vs 21k names, top-5 (BASELINE configs[1]): size-independent properties + oracle on a row sample."""
    cfg = synth.CONFIGS['C2']
    y = torch.randint(0, cfg.k, (cfg.n,), generator=torch.Generator().manual_seed(1))
    Xc, _ = synth.image_feats(cfg.n, cfg.k, cfg.seed + 500, y=y)
    Xc = synth.bf16_round(Xc)
    W = synth.vocabulary(cfg.v, cfg.seed + 900)
    vocab = naming.Vocabulary(W.cuda())
    fb = naming._feats_bf16(Xc)
    vals, idx, _, _ = naming.name_topk_raw(fb, vocab, 5, False)
    assert (vals[:, :-1] >= vals[:, 1:]).all()                               # sorted, largest first
    assert (idx >= 0).all() and (idx < cfg.v).all()
    assert (idx.sort(dim=1).values.diff(dim=1) != 0).all()                    # five distinct names per image
    v1, i1, _, _ = naming.name_topk_raw(fb, vocab, 1, False)                  # k=1 kernel == head of the k=5 list
    assert torch.equal(i1[:, 0], idx[:, 0]) and torch.equal(v1[:, 0], vals[:, 0])
    perm = torch.randperm(cfg.n, generator=torch.Generator().manual_seed(2)).cuda()
    vp, ip, _, _ = naming.name_topk_raw(fb[perm].contiguous(), vocab, 5, False)  # row-permutation equivariance
    assert torch.equal(ip, idx[perm]) and torch.equal(vp, vals[perm])
    rows = perm[:4096].cpu()
    _check_topk(vals[rows.cuda()], idx[rows.cuda()], Xc[rows], W, 5, 'ptsup', LOGIT_ATOL)
    # vote on the full result: counts of each cluster add up to rows * top_k
    names, counts, distinct, nrows, ovf = naming.vote_device(idx, y.numpy(), cfg.k, 5, 20)
    assert int(ovf) == 0 and int(nrows.sum()) == cfg.n
    assert (counts.sum(dim=1).cpu() <= nrows.cpu() * 5).all()
    c = 3
    co = naming_oracle.vote(idx.cpu(), y.numpy(), [c], 5)[c]
    assert _counter_list(co) == [(int(a), int(b)) for a, b in zip(names[c].cpu(), counts[c].cpu()) if a >= 0]


@pytest.mark.parametrize('softmax', [False, True])
def test_host_features_stream_in_chunks_and_equal_the_resident_launch(softmax):
    """score_topk on HOST features uploads wave-sized chunks under the kernel; rows are independent, so indices and
    logits must equal the single resident launch bit for bit (incl. the ragged last chunk).  The softmax denominator
    is summed per piece of the vocabulary sweep, and where a sweep is cut depends on the rows of the launch: the
    probabilities agree to fp32 rounding."""
    n, d, v = 2 * naming.STREAM_ROWS + 1111, 256, 3000
    g = torch.Generator().manual_seed(77)
    feats = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1)
    W = torch.nn.functional.normalize(torch.randn(v, d, generator=g), dim=1).t().contiguous()
    vocab = naming.Vocabulary(W)
    v_res, i_res = naming.score_topk(feats.cuda(), vocab, k=5, softmax=softmax)
    for host in (feats, feats.pin_memory(), feats.numpy()):
        v_str, i_str = naming.score_topk(host, vocab, k=5, softmax=softmax)
        assert torch.equal(i_str, i_res)
        assert torch.allclose(v_str, v_res, rtol=2e-6, atol=0) if softmax else torch.equal(v_str, v_res)


@pytest.mark.parametrize('n,v,d,k', [(40000, 11000, 64, 5), (40000, 300, 64, 1), (60000, 500, 40, 5), (40000, 5000, 512, 5),
                                     (127000, 100, 768, 1)])
def test_several_row_blocks_per_cta_pair_at_narrow_widths(n, v, d, k):
    """Regression: with one k-block per tile (D <= 64) and more than one work item per CTA pair the MMA issuers ran
    three tiles ahead of their parity waits and the pair deadlocked (found by tools/naming_stress.py).  Checked on a
    row sample against torch, margins as everywhere else."""
    g = torch.Generator().manual_seed(n + v + d)
    X = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).bfloat16()
    W = torch.nn.functional.normalize(torch.randn(v, d, generator=g), dim=1).bfloat16()
    vocab = naming.Vocabulary.from_rows(W.cuda())
    for _ in range(3):                                    # back to back, no sync in between
        vals, idx, _, _ = naming.name_topk_raw(X.cuda(), vocab, k, False)
    rows = torch.randperm(n, generator=g)[:1500]
    _check_topk(vals[rows.cuda()], idx[rows.cuda()], X[rows].float(), W.float().t().contiguous(), k, 'ptsup', LOGIT_ATOL)


@pytest.mark.parametrize('n,v,d,k', [(19000, 5000, 128, 1), (19000, 5000, 128, 5), (19000, 5000, 64, 5), (30000, 3000, 192, 5)])
def test_one_tile_work_items_at_narrow_widths_are_reproducible(n, v, d, k):
    """Regression (found by tools/naming_stress.py in round 2): the linear work partition leaves ONE-tile work items at the
    ends of a pair's range; with two k-blocks per tile (D = 128) an MMA issuer then meets a given k-block of an item only
    every third item, its early parity wait on the rows' barrier aliased with the fill before last, and about one launch
    in 10^4 scored a few rows against half-written operands.  300 back-to-back launches must equal the first bit for bit,
    and the first must equal torch on a row sample."""
    g = torch.Generator().manual_seed(n + v + d + k)
    X = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).bfloat16().cuda()
    W = torch.nn.functional.normalize(torch.randn(v, d, generator=g), dim=1).bfloat16()
    vocab = naming.Vocabulary.from_rows(W.cuda())
    plan = naming.TopKPlan(n, v, k, 'cuda')
    v0, i0, _, _ = plan.run(X, vocab, False)
    v0, i0 = v0.clone(), i0.clone()
    rows = torch.randperm(n, generator=g)[:1500]
    _check_topk(v0[rows.cuda()], i0[rows.cuda()], X[rows.cuda()].float().cpu(), W.float().t().contiguous(), k, 'ptsup', LOGIT_ATOL)
    bad = 0
    for rep in range(30):
        for _ in range(10):                                   # no sync inside a batch
            plan.run(X, vocab, False)
        torch.cuda.synchronize()
        bad += int((plan.idx != i0).sum()) + int((plan.vals != v0).sum())
    assert bad == 0
