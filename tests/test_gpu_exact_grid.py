"""Tie and NaN rules of the scoring top-k and the E-step argmin, pinned bit-exactly on exact-grid inputs.

Every entry of X, W and C is a / 8 with an integer |a| <= 3.  Such values are exact in bf16 (so the bf16 cast of the
scoring operands and the E-step's hi / lo split lose nothing: the lo plane is 0), and for D <= 768 every product and
every partial sum is a multiple of 1/64 far inside fp32's 24-bit significand.  The tensor cores' fp32 accumulation is
then exact in any summation order, so logits, distances, labels, top-k lists and the fp64 inertia must EQUAL a plain
float64 reference on every row - no margin mask, no unchecked share.  Grid data ties a lot by itself, and ties are
planted on purpose where the kernels cut their work: 32-column chunks, the two column halves of a scoring tile, 224-column
tiles, the pieces a row block is cut into between CTA pairs, vocabulary shards, 256-column centroid tiles.

The reference order is explicit: top-k = stable descending sort (value descending, lower column first; torch.topk does
not promise that order among equal values); argmin = first minimum, and the first NaN when a row has one (what torch.min
returns on the CPU).  Softmax probabilities keep the suite's 1e-5 tolerance; their indices are exact."""
import numpy as np
import pytest
import torch

from scd_b200 import _lib, dist as sdist, kmeans, naming

SCALE = 100.0
P_ATOL = 1e-5
MAX_D = 768


def _grid(shape, g, density=0.3):
    """Sparse grid values a / 8, a in {-3 .. 3} \\ {0} on about `density` of the entries."""
    a = torch.randint(1, 4, shape, generator=g) * (torch.randint(0, 2, shape, generator=g) * 2 - 1)
    return (a * (torch.rand(shape, generator=g) < density)).float() / 8


def _dense_grid(d, g):
    """A dense vector of +-3/8: the largest norm on the grid, so x . w < x . x for every grid column w != x."""
    return (torch.randint(0, 2, (d,), generator=g) * 2 - 1).float() * 3 / 8


def test_grid_inputs_are_exact():
    """The premise of this file, checked once without a GPU: grid values are bf16-exact with a zero lo plane, and the
    largest dot product and squared distance at D = 768 are multiples of 1/64 that fp32 holds exactly, also scaled by 100."""
    g = torch.Generator().manual_seed(0)
    x = _grid((4096, MAX_D), g)
    assert torch.equal(x.bfloat16().float(), x) and torch.equal((x - x.bfloat16().float()).bfloat16().float(), torch.zeros_like(x))
    assert 0.25 < float((x != 0).float().mean()) < 0.35
    assert float(x.abs().max()) == 3 / 8 and torch.equal(x * 8, (x * 8).round())
    max_dot = MAX_D * 3 * 3                       # |m| of a dot product m / 64
    max_sq = MAX_D * 6 * 6                        # |m| of a squared distance m / 64
    assert max_dot == 6912 and max_sq == 27648
    for m in (max_dot, max_dot - 1, max_sq, max_sq - 1):
        assert float(torch.tensor(m / 64, dtype=torch.float32)) * 64 == m
        assert float(torch.tensor(SCALE, dtype=torch.float32) * torch.tensor(m / 64, dtype=torch.float32)) == SCALE * m / 64
    # the fp64 inertia of 148 * 128 * 2 + 77 rows at the largest distance is exact too
    assert (37965 * max_sq) < 2 ** 53
    u, w = _dense_grid(MAX_D, g), x[0]
    assert float(u @ u) > float(u @ w) and float(u @ u) == 9 * MAX_D / 64


# ------------------------------------------------------------------------------------------------ scoring top-k
def _ref_topk(X, W, k):
    """fp64 logits (exact here) -> (top-k logits, indices) in (value descending, column ascending) order; also
    returns the (k+1)-th column of the sorted logits so the caller can see the ties at the k-th position."""
    L = X.double().cuda() @ W.double().cuda()
    s = torch.sort(L, dim=1, descending=True, stable=True)
    kk = min(k + 1, W.shape[1])
    return L, s.values[:, :kk], s.indices[:, :kk]


def _ref_softmax(L, idx):
    lm = L.max(dim=1, keepdim=True).values
    e = torch.exp(SCALE * (L - lm))
    return (e.gather(1, idx) / e.sum(dim=1, keepdim=True)), lm.view(-1), e.sum(dim=1)


def _tie_share(vals, k):
    """rows with two equal values inside the sorted top-(k+1)"""
    if vals.shape[1] < 2:
        return 0.0
    return float((vals[:, :-1] == vals[:, 1:]).any(dim=1).float().mean())


def _plan(n, v, k):
    out = np.zeros(6, dtype=np.int32)
    _lib.check(_lib.load().scd_name_topk_plan(n, v, k, out.ctypes.data), 'scd_name_topk_plan')
    return out


def _first_cut(n, v, k):
    """(row block, first tile) of the first work item that starts inside a row block (t0 > 0): there the row block is
    cut between two CTA pairs and the merge joins the pieces."""
    lib = _lib.load()
    items = np.zeros((4096, 4), dtype=np.int32)
    for pair in range(int(_plan(n, v, k)[2])):
        got = lib.scd_name_topk_plan_pair(n, v, k, pair, items.ctypes.data, items.shape[0])
        assert got >= 0
        for rb, t0, _nt, _part in items[:got]:
            if t0 > 0:
                return int(rb), int(t0)
    raise AssertionError('no row block is cut')


def _planted(n, v, d, k_max, seed):
    """Grid features [n, d] and vocabulary [d, v] with exact ties planted at the boundaries of the kernel's work:
    probe rows x = u (dense +-3/8) and copies of u as vocabulary columns, so the probe's best logits are those copies.
    Returns (X, W, probe rows)."""
    g = torch.Generator().manual_seed(seed)
    X, W = _grid((n, d), g), _grid((d, v), g)
    rb, t0 = _first_cut(n, v, k_max)
    cut = t0 * 224
    sets = [                                            # the first three never share a column, later ones may be dropped
        ([cut - 1, cut], rb),                           # a row block cut between two CTA pairs
        ([int(p) for p in np.linspace(1, v - 3, k_max + 1)], None),     # k + 1 equal copies: only the k lowest appear
        ([3 + 8 * j for j in range(25)] + [v - 5], None),               # > KT + 4 maxima, spread over chunks: the drain loop
        ([31, 32], None),                               # chunk boundary
        ([127, 128], None),                             # column halves of a tile
        ([223, 224], None),                             # tile boundary
        ([v - 2, v - 1], None),                         # ragged last tile
        ([100, 37, 2, 500, 260], None),                 # pushed out of column order
    ]
    probes, taken = [], set()
    rows = torch.randperm(n, generator=g).tolist()
    for j, (cols, in_block) in enumerate(sets):
        if taken & set(cols):
            assert j >= 3
            continue
        taken |= set(cols)
        u = _dense_grid(d, g)
        W[:, cols] = u.view(-1, 1)
        for rep in range(3):
            r = in_block * 256 + (1 + rep * 97 + j) % min(256, n - in_block * 256) if in_block is not None else rows.pop()
            X[r] = u
            probes.append(r)
    # all-zero feature rows: every logit is 0, the answer is columns 0 .. k-1
    for r in (0, n - 1, rows.pop()):
        X[r] = 0
        probes.append(r)
    return X, W, sorted(set(probes))


# share of rows with a tie inside the top-(k+1) that grid data guarantees (measured: about twice these at D = 768)
MIN_TIE_SHARE = {1: 0.015, 2: 0.05, 5: 0.2, 6: 0.25, 8: 0.35}


def _check_scoring(X, W, k, softmax, probes):
    """One launch (softmax: with the row statistics) against the reference: indices and logits / row maxima exact."""
    v = W.shape[1]
    L, rv, ri = _ref_topk(X, W, k)
    kk = min(k, v)
    assert _tie_share(rv, k) >= MIN_TIE_SHARE[k]
    assert _tie_share(rv[probes], k) == 1.0
    vocab = naming.Vocabulary(W.cuda())
    fb = naming._feats_bf16(X)
    assert torch.equal(fb.float(), X.cuda())
    vals, idx, rmax, rsum = naming.name_topk_raw(fb, vocab, k, softmax, want_stats=softmax)
    assert torch.equal(idx, ri[:, :kk]), int((idx != ri[:, :kk]).any(dim=1).sum())
    if softmax:
        p, lm, es = _ref_softmax(L, ri[:, :kk])
        assert torch.allclose(vals.double(), p, atol=P_ATOL, rtol=0)
        assert torch.equal(rmax, lm.float())
        assert torch.allclose(rsum.double(), es, rtol=P_ATOL, atol=0)
    else:
        assert torch.equal(vals, (SCALE * rv[:, :kk]).float())
    return vals, idx


@pytest.mark.gpu
@pytest.mark.parametrize('n,v,d', [(600, 2500, 64), (600, 2500, 72), (600, 2500, 768), (19000, 5000, 128), (4000, 21000, 768)])
def test_scoring_topk_ties_on_the_grid(n, v, d):
    """Every list length and both merge forms (k = 1 / 2 / 5 / 6 / 8: lists of 1, 5, 8; 2 and 6 take the merge that does
    not fill its whole list), with and without softmax, on a small launch (every row block cut into single tiles), a
    multi-item launch and a C2-width launch; indices, logits and row maxima exact."""
    X, W, probes = _planted(n, v, d, 8, seed=n + v + d)
    for k in (1, 2, 5, 6, 8):
        assert int(_plan(n, v, k)[3]) >= 2                           # some row block is really cut between CTA pairs
        for softmax in (False, True):
            _check_scoring(X, W, k, softmax, probes)
    # the zero rows: columns 0 .. k-1
    vals, idx, _, _ = naming.name_topk_raw(naming._feats_bf16(X[[0, n - 1]]), naming.Vocabulary(W.cuda()), 8, False)
    assert idx.tolist() == [list(range(8))] * 2 and not vals.any()


@pytest.mark.gpu
@pytest.mark.parametrize('k', [1, 5, 6])
def test_vocabulary_shards_merge_ties_across_shard_bounds(k):
    """Three vocabulary shards with tied copies on both sides of each shard bound: the merged lists equal the unsharded
    lists and the reference, with and without softmax."""
    n, v, d = 3000, 4099, 128
    g = torch.Generator().manual_seed(40 + k)
    X, W = _grid((n, d), g), _grid((d, v), g)
    bounds = [sdist.shard_bounds(v, 3, r) for r in range(3)]
    probes = []
    for lo, _hi in bounds[1:]:
        for cols in ([lo - 1, lo], [lo - 3, lo - 2] + [lo + 1 + 7 * j for j in range(k)], [lo - 301, lo + 300]):
            u = _dense_grid(d, g)
            W[:, cols] = u.view(-1, 1)
            rows = [100 * (len(probes) // 4 + 1) + rep for rep in range(4)]
            X[rows] = u
            probes += rows
    X[7] = 0
    probes.append(7)
    fb = naming._feats_bf16(X)
    for softmax in (False, True):
        want_v, want_i = _check_scoring(X, W, k, softmax, probes)
        parts = []
        for lo, hi in bounds:
            vocab = naming.Vocabulary(W[:, lo:hi].cuda(), col_offset=lo)
            parts.append(naming.name_topk_raw(fb, vocab, k, False, want_stats=True))
        got_v, got_i = sdist.merge_topk_parts(parts, k, softmax)
        assert torch.equal(got_i, want_i)
        if softmax:
            assert torch.allclose(got_v, want_v, atol=P_ATOL, rtol=0)
        else:
            assert torch.equal(got_v, want_v)
    assert got_i[7].tolist() == list(range(k))


@pytest.mark.gpu
def test_reassign_and_clip_preds_take_the_first_of_equal_names():
    """A candidate list that names one column twice ([5, 9, 5]) and a vocabulary with duplicated columns: argmax returns
    the first maximum, so a repeated name never wins at its later position."""
    n, v, d = 2000, 300, 64
    g = torch.Generator().manual_seed(9)
    X, W = _grid((n, d), g), _grid((d, v), g)
    W[:, 9] = -W[:, 5]
    X[:50] = 0                                                        # every candidate ties
    X[50:100] = W[:, 5]                                               # the copies of column 5 tie at the top
    for cand in ([5, 9, 5], [9, 5, 9, 5]):
        got = naming.reassign(X, W, cand)
        L = X.double() @ W[:, cand].double()
        want = torch.sort(L, dim=1, descending=True, stable=True).indices[:, 0].numpy()
        assert np.array_equal(got, want)
        assert not np.isin(got, [j for j, c in enumerate(cand) if c in cand[:j]]).any()
        assert (got[:50] == 0).all() and (got[50:100] == cand.index(5)).all()
    u = _dense_grid(d, g)
    W[:, [17, 200, 250]] = u.view(-1, 1)
    X[100:150] = u
    L = X.double() @ W.double()
    want = torch.sort(L, dim=1, descending=True, stable=True).indices[:, 0]
    got = naming.clip_preds(X, W).cpu()
    assert torch.equal(got, want) and (got[100:150] == 17).all() and (got[:50] == 0).all()


# ------------------------------------------------------------------------------------------------ E-step
def _ref_dist(X, C):
    """plain fp64 sum_d (x - c)^2 on the device, in row chunks"""
    Xd, Cd = X.double().cuda(), C.double().cuda()
    step = max(1, (1 << 27) // max(1, C.shape[0] * C.shape[1]))
    return torch.cat([((Xd[i:i + step, None, :] - Cd[None]) ** 2).sum(-1) for i in range(0, X.shape[0], step)])


def _ref_argmin(dist):
    """torch.min's rule: the first NaN of a row if it has one, else the first minimum"""
    nan = dist.isnan()
    m = dist.masked_fill(nan, float('inf')).min(dim=1).values
    first_min = (dist == m[:, None]).int().argmax(dim=1)
    has_nan = nan.any(dim=1)
    return torch.where(has_nan, nan.int().argmax(dim=1), first_min), torch.where(has_nan, torch.full_like(m, float('nan')), m)


def _same(a, b):
    """equal values (-0 == +0), NaN exactly where the other has NaN"""
    a, b = a.double().cpu(), b.double().cpu()
    na, nb = a.isnan(), b.isnan()
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


def _estep_case(n, d, k, far, seed):
    """Grid X [n, d] and C [k, d] with duplicate centroids, rows on duplicated centroids (distance exactly 0) and rows at
    the midpoint of two centroids that differ by 2/8 in one coordinate.  The duplicates sit inside one 32-column chunk
    (5/6), on both sides of a chunk (31/32) and of a centroid tile (255/256), and at the end (K-2/K-1) - or, with `far`,
    at both ends (3/K-1).  Returns (X, C, tie rows)."""
    g = torch.Generator().manual_seed(seed)
    X, C = _grid((n, d), g), _grid((k, d), g)
    dups = [(a, b) for a, b in ((5, 6), (31, 32), (255, 256), (3, k - 1) if far else (k - 2, k - 1)) if a < b < k]
    dups = [p for i, p in enumerate(dups) if not set(p) & {x for q in dups[:i] for x in q}]
    used = {x for p in dups for x in p}
    mids = []
    for a, b in ((7, 8), (0, 9), (30, 33), (200, 300), (1, k - 3), (250, 257)):
        if a < b < k and not {a, b} & used:
            mids.append((a, b))
            used |= {a, b}
    for a, b in dups:
        C[b] = C[a]
    for a, b in mids:
        j = (a * 7 + b) % d
        C[b] = C[a]
        C[a, j], C[b, j] = -1 / 8, 1 / 8
    rows = torch.randperm(n, generator=g).tolist()
    tie_rows = []
    for a, b in dups + mids:
        for _ in range(n // (10 * len(dups + mids))):
            r = rows.pop()
            X[r] = C[a]
            if (a, b) in mids:
                X[r, (a * 7 + b) % d] = 0
            tie_rows.append(r)
    return X, C, tie_rows


def _run_estep(X, C, exact):
    labels = torch.empty(X.shape[0], dtype=torch.int64, device='cuda')
    mind = torch.empty(X.shape[0], dtype=torch.float32, device='cuda')
    acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    kmeans._estep(X.cuda(), C.cuda(), labels, acc, mind, exact=exact)
    return labels, mind, acc


def _check_estep(X, C, paths, tie_rows=()):
    """The E-step on each path (exact=False / True) against the fp64 reference: labels, distances and inertia equal.
    Returns the reference (distances, labels)."""
    dist = _ref_dist(X, C)
    want_l, want_m = _ref_argmin(dist)
    if len(tie_rows):                                                 # the planted ties are there
        t = dist[torch.tensor(tie_rows)]
        assert ((t == t.min(dim=1, keepdim=True).values).sum(dim=1) >= 2).all()
    for exact in paths:
        labels, mind, acc = _run_estep(X, C, exact)
        assert torch.equal(labels, want_l), (exact, int((labels != want_l).sum()))
        assert _same(mind, want_m), exact
        assert _same(acc, want_m.sum().view(1)), exact
    return dist, want_l


def check_estep_grid(k, d):
    """Every E-step path (D = 32 / 36: the fp32 direct-form kernel only; D >= 40: the tensor-core kernel and exact=True) and
    pairwise_distance equal the fp64 reference on grid data with planted ties and NaNs: labels (ties -> lowest k, a NaN
    distance wins, the first NaN of several), distances and inertia (NaN exactly where the reference's are)."""
    n = 148 * 128 * 2 + 77 if k > 256 else 4000 + k
    tc = d >= 40
    assert _lib.load().scd_estep_uses_tensor_cores(n, d, k) == int(tc)
    paths = (False, True) if tc else (False,)
    for far in (False, True):
        X, C, tie_rows = _estep_case(n, d, k, far, seed=k * 1000 + d + far)
        assert len(tie_rows) >= n // 20
        dist, want = _check_estep(X, C, paths, tie_rows)
        got = kmeans.pairwise_distance(X.cuda(), C.cuda())
        assert torch.equal(got.double(), dist)
    # NaN centroids: one at a chunk / tile edge, one with a single NaN coordinate, two in one chunk, two in different
    # chunks.  The numeric best of most rows lies before or after the NaN, in the same or in another centroid tile.
    nan_sets = [[p] for p in (0, 31, 32, 255, 256, k - 1) if p < k] + [[(k // 3, d - 1)], [10, 11], [k // 2, k - 1]]
    for nan_cols in nan_sets:
        Cn = C.clone()
        for p in nan_cols:
            Cn[p] = float('nan')                                      # a whole row, or the one entry (k, j)
        _, want = _check_estep(X, Cn, paths)
        first = min(p[0] if isinstance(p, tuple) else p for p in nan_cols)
        assert (want == first).all()
    # a NaN entry in a row of X: every distance of that row is NaN -> label 0, NaN distance
    bad = [1, n // 2, n - 1]
    X[bad, d // 2] = float('nan')
    _, want = _check_estep(X, C, paths)
    assert (want[bad] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize('k,d', [(k, d) for d in (40, 768) for k in (12, 160, 161, 200, 256, 257, 1000, 1024)])
def test_estep_ties_and_nan_on_the_grid(k, d):
    """Tensor-core E-step: TMEM operand for K <= 160 at D = 768, shared-memory operand otherwise, the ragged 16-column
    chunk at K = 161, several 256-column centroid tiles for K > 256; and the fp32 direct-form kernel (exact=True) on the
    same inputs.  (D = 32 / 36, where only the direct-form kernel runs: test_gpu_kmeans.test_estep_tie_and_nan_rules.)"""
    check_estep_grid(k, d)
