"""GPU parity at the sizes and code paths the small-shape tests do not reach (VERDICT round 1, "Weak #1"):

  * E-step with several centroid tiles per row tile (K > 256: C5's K = 1000, the shared-memory-A variant) and the
    160 < K <= 256 shared-memory variant, on multi-tile persistent launches, against the oracle on a row sample;
  * C1 (6 000 x 768, K = 200, V = 11 000 - the config the CPU oracle runs IN FULL): one whole round, k-means iteration,
    top-5 and voted names, against the oracle;
  * scoring / top-k at V = 82 000 and V = 100 000 with several waves of row blocks plus a vocabulary-split tail wave,
    against the oracle on a row sample, and as a size-independent property (shard-and-merge of the vocabulary gives the
    same lists);
  * the vote at N = 1.28 M, K = 1000 and for clusters beyond the shared-memory table (global spill tables);
  * the operands scd_finalize_centers leaves for the next E-step are the ones the E-step derives itself.

Tolerances as in test_gpu_kmeans.py / test_gpu_naming.py (written there): distances 1e-4, labels exact where the
top-1 / top-2 margin > 1e-5, logits 2e-3 on the x100 scale, indices exact where the neighbouring gaps > 1e-3."""
import numpy as np
import pytest
import torch

from oracle import kmeans_oracle, naming_oracle
from scd_b200 import dist as sdist, kmeans, naming, synth

pytestmark = pytest.mark.gpu
TAU_D, ATOL_D = 1e-5, 1e-4
TAU_L, ATOL_L = 1e-3, 2e-3


def _sample_rows(n, m, seed):
    g = torch.Generator().manual_seed(seed)
    head = torch.arange(min(256, n))
    tail = torch.arange(max(n - 256, 0), n)
    rnd = torch.randint(0, n, (m,), generator=g)
    return torch.unique(torch.cat((head, tail, rnd)))


@pytest.mark.parametrize('k,d', [(257, 768), (512, 768), (1000, 768), (1024, 512), (1000, 512), (200, 768), (256, 512)])
def test_estep_many_centroid_tiles_against_oracle(k, d):
    n = 148 * 128 * 2 + 77                        # two full waves of 128-row tiles on 148 SMs + a ragged tile
    g = torch.Generator().manual_seed(k + d)
    mu = synth.unit_rows(torch.randn(k, d, generator=g))
    X = synth.unit_rows(torch.randn(n, d, generator=g) + 3.0 * mu[torch.randint(0, k, (n,), generator=g)])
    C = synth.unit_rows(mu + 0.05 * torch.randn(k, d, generator=g))
    Xd, Cd = X.cuda(), C.cuda()
    labels = torch.empty(n, dtype=torch.int64, device='cuda')
    mind = torch.empty(n, dtype=torch.float32, device='cuda')
    acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    kmeans._estep(Xd, Cd, labels, acc, mind)
    rows = _sample_rows(n, 1536, k)
    ref = kmeans_oracle.pairwise_distance(X[rows], C, 256)
    two = ref.topk(2, dim=1, largest=False).values
    ok = (two[:, 1] - two[:, 0]) > TAU_D
    assert ok.float().mean() > 0.98
    assert torch.equal(labels.cpu()[rows][ok], ref.argmin(dim=1)[ok])
    assert torch.allclose(mind.cpu()[rows], ref.min(dim=1).values, atol=ATOL_D, rtol=0)
    # size-independent: the tensor-core E-step and the fp32 direct-form kernel agree on every row with a clear margin,
    # and the inertia is the sum of the minima
    exact, mind_x = torch.empty_like(labels), torch.empty_like(mind)
    kmeans._estep(Xd, Cd, exact, None, mind_x, exact=True)
    assert torch.allclose(mind, mind_x, atol=ATOL_D, rtol=0)
    differ = labels != exact
    if differ.any():
        dd = kmeans.pairwise_distance(Xd[differ], Cd)
        two = dd.topk(2, dim=1, largest=False).values
        assert float((two[:, 1] - two[:, 0]).max()) <= TAU_D
    assert abs(acc.item() - mind.double().sum().item()) < 1e-6 * n
    # back-to-back launches reproduce the first one bit for bit (ring / parity state carries nothing over)
    again = torch.empty_like(labels)
    for _ in range(3):
        kmeans._estep(Xd, Cd, again, None)
        assert torch.equal(again, labels)


def test_finalize_leaves_the_next_esteps_operands():
    """scd_finalize_centers(estep_ws=...) leaves the same workspace bytes (hi / lo planes, ||c||^2) as the E-step's own
    split of the new centres, and with SCD_ESTEP_PLANES_READY gives bit-identical labels / distances - including a NaN
    centre (empty cluster)."""
    cfg = synth.Config('t', 20000, 100, 10, 11)
    data = synth.make(cfg, d=768)
    X, C0 = data['X'].cuda(), data['C0'].cuda()
    n, k, d = X.shape[0], cfg.k, X.shape[1]
    ms, es = kmeans._MStep(n, d, k, 'cuda'), kmeans._EStep(k, d, 'cuda')
    labels = torch.empty(n, dtype=torch.int64, device='cuda')
    es.run(X, C0, labels, None)
    labels[labels == 7] = 8                                   # cluster 7 becomes empty -> NaN centre
    ms.sums_counts(X, labels)
    c_new = torch.empty_like(C0)
    ms.finalize(C0, c_new, estep=es, shift=False)
    assert es.ready_for == c_new.data_ptr() and torch.isnan(c_new[7]).all()
    ws_finalize = es.ws.clone()
    l1, m1 = torch.empty_like(labels), torch.empty(n, device='cuda')
    es.run(X, c_new, l1, None, m1)                            # uses the operands finalize left behind
    assert es.ready_for is None
    l2, m2 = torch.empty_like(labels), torch.empty(n, device='cuda')
    kmeans._estep(X, c_new, l2, None, m2)                     # splits c_new itself
    assert torch.equal(l1, l2) and torch.equal(m1.isnan(), m2.isnan()) and torch.equal(m1[~m1.isnan()], m2[~m2.isnan()])
    assert (l1 == 7).all()                                    # torch.min: a NaN distance beats any number
    es.ready_for = None
    es.run(X, c_new, l2, None)                                # centroid_split_kernel rewrites es.ws from c_new
    assert torch.equal(es.ws, ws_finalize)                    # byte for byte, the NaN row of cluster 7 included
    # the host-side sum of the move norms is the device-side shift
    ms.finalize(C0, c_new)
    assert torch.equal(torch.isnan(ms.shift), torch.isnan(ms.norms[:k].sum().view(1)))


def test_c1_full_round_against_the_oracle():
    """C1 end to end at full size (the CPU-runnable config): k-means iteration, scoring + top-5, vote, voted candidates."""
    cfg = synth.CONFIGS['C1']
    data = synth.make(cfg)
    X, Xc, W, C0 = data['X'], data['Xc'], data['W'], data['C0']
    # ---- k-means iteration
    lab_o, mind_o, inertia_o = kmeans_oracle.estep(X, C0.clone(), 1024)
    cen_o = kmeans_oracle.mstep(X, lab_o, C0.clone())
    km = kmeans.K_Means(k=cfg.k, max_iterations=1, init='first', n_init=1)
    Xd = X.cuda()
    labels, inertia, centers, _ = km._lloyd(Xd, Xd, torch.empty(cfg.n, dtype=torch.int64, device='cuda'), 0, C0.cuda())
    dist = kmeans_oracle.pairwise_distance(X, C0, 1024)
    two = dist.topk(2, dim=1, largest=False).values
    clear = (two[:, 1] - two[:, 0]) > TAU_D
    assert clear.float().mean() > 0.999
    assert torch.equal(labels.cpu()[clear], lab_o[clear])
    assert abs(float(inertia) - float(inertia_o)) < 1e-6 * cfg.n
    if torch.equal(labels.cpu(), lab_o):
        assert torch.allclose(centers.cpu(), cen_o, atol=ATOL_D, rtol=1e-5, equal_nan=True)
    # ---- scoring + top-5 (both drivers' variants)
    for variant, softmax, atol in (('ptsup', False, ATOL_L), ('unsup', True, 1e-5)):
        idx_o, val_o = naming_oracle.score_topk(Xc, W, 6, variant=variant)
        vals, idx = naming.score_topk(Xc, W, k=5, softmax=softmax)
        assert torch.allclose(vals.cpu(), val_o[:, :5], atol=atol, rtol=1e-4 if softmax else 0)
        lv = naming_oracle.score_topk(Xc, W, 6, variant='ptsup')[1]
        gaps = (lv[:, :-1] - lv[:, 1:]) > TAU_L
        left = torch.cat((torch.ones(cfg.n, 1, dtype=torch.bool), gaps[:, :4]), dim=1)
        pinned = left & gaps
        assert pinned.float().mean() > 0.97
        assert torch.equal(idx.cpu()[pinned], idx_o[:, :5][pinned])
    # ---- vote + candidates on the oracle's own labels / indices (bit-exact: integer work)
    idx_o5 = naming_oracle.score_topk(Xc, W, 5, variant='ptsup')[0]
    ids = list(range(cfg.k))
    c2c_o = naming_oracle.vote(idx_o5, lab_o.numpy(), ids, 5)
    c2c = naming.vote(idx_o5, lab_o.numpy(), ids, 5, 20)
    for c in ids:
        assert [(int(a), int(b)) for a, b in c2c[c].most_common(20)] == [(int(a), int(b)) for a, b in c2c_o[c].most_common(20)]
    uniq_o = naming_oracle.voted_candidates(c2c_o, ids, 20)
    assert naming.voted_candidates(c2c, ids, 20) == uniq_o
    ind_o, w_o = naming_oracle.assign_name(uniq_o, c2c_o, num_common=4)
    ind, w = naming.assign_name(uniq_o, c2c, num_common=4)
    assert np.array_equal(w, w_o) and np.array_equal(ind, ind_o)
    # ---- and the whole device round from the device's own labels / indices: voted names equal the oracle's wherever
    # its inputs (labels, top-5 indices) are the oracle's
    vals, idx = naming.score_topk(Xc, W, k=5, softmax=False)
    if torch.equal(idx.cpu(), idx_o5) and torch.equal(labels.cpu(), lab_o):
        names, counts, _, _, ovf = naming.vote_device(idx, labels, cfg.k, 5, 20)
        assert int(ovf.item()) == 0
        for c in ids:
            want = [(int(a), int(b)) for a, b in c2c_o[c].most_common(20)]
            got = [(int(a), int(b)) for a, b in zip(names[c].tolist(), counts[c].tolist()) if a >= 0]
            assert got == want


@pytest.mark.parametrize('v,n', [(82_000, 74 * 256 * 4 + 13 * 256 + 5), (100_000, 74 * 256 * 2 + 60 * 256 + 255)])
def test_scoring_big_vocabulary_multi_wave(v, n):
    """many row blocks per CTA pair, most swept whole and some cut between two pairs (int32 ranges, big gathers)"""
    g = torch.Generator().manual_seed(v)
    plan = np.zeros(6, dtype=np.int32)
    from scd_b200 import _lib
    _lib.check(_lib.load().scd_name_topk_plan(n, v, 5, plan.ctypes.data), 'plan')
    assert plan[0] >= 2 * plan[2] and plan[3] == 2           # whole-vocabulary items AND row blocks cut between two pairs
    feats = torch.empty(n, 768)
    for lo in range(0, n, 65536):
        hi = min(lo + 65536, n)
        feats[lo:hi] = synth.bf16_round(synth.unit_rows(torch.randn(hi - lo, 768, generator=g)))
    W = synth.vocabulary(v, seed=v)
    vocab = naming.Vocabulary(W.cuda())
    fb = naming._feats_bf16(feats)
    vals, idx, _, _ = naming.name_topk_raw(fb, vocab, 5, False)
    rows = _sample_rows(n, 768, v)
    oi, ov = naming_oracle.score_topk(feats[rows], W, 6, variant='ptsup')
    assert torch.allclose(vals.cpu()[rows], ov[:, :5], atol=ATOL_L, rtol=0)
    gaps = (ov[:, :-1] - ov[:, 1:]) > TAU_L
    left = torch.cat((torch.ones(len(rows), 1, dtype=torch.bool), gaps[:, :4]), dim=1)
    pinned = left & gaps
    assert pinned.float().mean() > 0.97
    assert torch.equal(idx.cpu()[rows][pinned], oi[:, :5][pinned])
    assert int(idx.min()) >= 0 and int(idx.max()) < v
    # size-independent properties over ALL rows: values sorted, indices distinct per row, a second launch is bit-identical,
    # and scoring three vocabulary shards + k-way merge reproduces the lists
    assert bool((vals[:, :-1] >= vals[:, 1:]).all())
    srt = idx.sort(dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())
    vals2, idx2, _, _ = naming.name_topk_raw(fb, vocab, 5, False)
    assert torch.equal(idx2, idx) and torch.equal(vals2, vals)
    parts = []
    for r in range(3):
        lo, hi = sdist.shard_bounds(v, 3, r)
        parts.append(naming.name_topk_raw(fb, naming.Vocabulary.from_rows(vocab.Wt[lo:hi], col_offset=lo), 5, False, want_stats=True))
    mv, mi = sdist.merge_topk_parts(parts, 5, False)
    assert torch.equal(mi, idx) and torch.allclose(mv, vals, atol=1e-5, rtol=0)


def _check_vote(names, counts, idx, preds, clusters, top_k, m):
    co = naming_oracle.vote(idx, preds, clusters, top_k)
    names, counts = names.cpu().numpy(), counts.cpu().numpy()
    for c in clusters:
        want = [(int(a), int(b)) for a, b in co[c].most_common(m)]
        got = [(int(a), int(b)) for a, b in zip(names[c], counts[c]) if a >= 0]
        assert got == want, c


def test_vote_at_c5_size():
    """N = 1.28 M rows, K = 1000 clusters, names drawn with a heavy head so counts tie a lot; checked against the oracle's
    Counter on a sample of clusters, the row counts on all of them."""
    g = torch.Generator().manual_seed(12)
    n, k, v = 1_280_000, 1000, 100_000
    preds = torch.randint(0, k, (n,), generator=g)
    idx = (torch.rand(n, 5, generator=g) ** 6 * v).long().clamp_(max=v - 1)
    names, counts, distinct, rows, ovf = naming.vote_device(idx.cuda(), preds.cuda(), k, 5, 20)
    assert int(ovf.item()) == 0
    assert torch.equal(rows.cpu().long(), torch.bincount(preds, minlength=k))
    clusters = [0, 1, 17, 499, 998, 999]
    _check_vote(names, counts, idx, preds.numpy(), clusters, 5, 20)
    for c in clusters:
        assert int(distinct[c]) == len(set(idx[preds == c].reshape(-1).tolist()))
    # the packed int32 records of the multi-GPU path give the same result
    rec = naming.pack_vote_records(preds.cuda(), idx.cuda(), 5)
    assert rec.dtype == torch.int32 and rec.shape == (n, 6)
    n2, c2, d2, r2, o2 = naming.vote_records(rec, k, 20)
    assert torch.equal(n2, names) and torch.equal(c2, counts) and torch.equal(d2, distinct) and torch.equal(r2, rows)


@pytest.mark.parametrize('known', [None, [3, 5, 70_000]])
def test_vote_clusters_beyond_the_shared_memory_table(known):
    """127 k rows in 3 clusters: ~42 k rows x 5 names per cluster, > 16 384 distinct names each - the histogram is built
    in the global spill tables (round 1 raised an overflow error here)."""
    g = torch.Generator().manual_seed(13)
    n, k, v = 127_000, 3, 90_000
    preds = torch.randint(0, k, (n,), generator=g)
    preds[:5] = 2
    idx = torch.randint(0, v, (n, 5), generator=g)
    idx[:, 0] = torch.randint(0, 50, (n,), generator=g)
    # also on the label sort the M-step has just made (scd_vote_presorted): that sort is not stable, the vote's
    # first-occurrence tie order must not depend on it
    ms = kmeans._MStep(n, 4, k, 'cuda')
    ms.sums_counts(torch.randn(n, 4, generator=torch.Generator().manual_seed(14)).cuda(), preds.cuda())
    co = naming_oracle.vote(idx, preds.numpy(), list(range(k)), 5, known_name_idx=known)
    for presorted in (None, ms):
        names, counts, distinct, rows, ovf = naming.vote_device(idx.cuda(), preds.cuda(), k, 5, 20, known, presorted=presorted)
        assert int(ovf.item()) == 0 and int(distinct.min()) > 16384
        assert torch.equal(rows.cpu().long(), torch.bincount(preds, minlength=k))
        for c in range(k):
            want = [(int(a), int(b)) for a, b in co[c].most_common(20)]
            got = [(int(a), int(b)) for a, b in zip(names[c].tolist(), counts[c].tolist()) if a >= 0]
            assert got == want
            assert int(distinct[c]) == len(co[c])
    # top_k = 2 of the same lists, and many ties at the selection threshold (every name seen once or twice)
    idx2 = torch.randperm(n * 5, generator=g).view(n, 5) % 200_000
    for presorted in (None, ms):
        names, counts, _, _, ovf = naming.vote_device(idx2.cuda(), preds.cuda(), k, 2, 20, presorted=presorted)
        assert int(ovf.item()) == 0
        _check_vote(names, counts, idx2, preds.numpy(), list(range(k)), 2, 20)
