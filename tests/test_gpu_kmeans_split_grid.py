"""The k-means pass pinned bit-exactly on two-plane grid inputs: the E-step's hi / lo split, the M-step's sums and centres,
the labelled inertia, k-means++ and the int32 cost matrix.

Every entry of X and C is a / 8 + b / 2^11 with |a| in {2, 3} and b in {-1, 0, 1}, or a = +-1 with b = 0 (for |a| = 1,
2^-11 is a rounding tie of the bf16 cast).  Torch's round-to-nearest bf16 split then gives exactly hi = a / 8 and
lo = b / 2^11, so the lo plane is NOT zero (about two thirds of the entries carry one), and the E-step's documented form
    dist = ||x||^2 + ||c||^2 - 2 (x_hi . c_hi + x_hi . c_lo + x_lo . c_hi)
differs from the true distance by 2 x_lo . c_lo.  Rows have at most NNZ = 7 non-zero entries, so every row r has
S(r) = sum_d (|r_hi| + |r_lo|)^2 <= 7 (3/8 + 2^-11)^2 < 1, and then:
  * products: hi.hi is a multiple of 2^-6, hi.lo of 2^-14, x^2 of 2^-22;
  * every partial sum of the MMA accumulator is at most sqrt(S(x) S(c)) <= 1 in magnitude (Cauchy-Schwarz) on the 2^-14
    grid: 15 bits;
  * fma(-2, acc, ||c||^2) is at most 3 in magnitude on the 2^-22 grid (24 bits), the final distance at most 4 = 2^24 units;
so everything is exact in fp32 in any summation order, and the fp64 inertia of N <= 2^27 rows is exact too.  The kernels
must therefore EQUAL a plain fp64 evaluation of what they document, on every row, with no margin mask.  For the M-step the
bound is sum |x| < 2^13 per (cluster, column), on the 2^-11 grid: the sums are exact whatever order the label sort and the
vector atomics add the rows in.

Centroid pairs are planted so that the hi-only distances tie and the lo terms decide the label (kinds A, B, C below);
test_split_grid_premise shows, on the reference side, that each part of the split changes the result on this data."""
import numpy as np
import pytest
import torch

from scd_b200 import _lib, kmeans

E = 2.0 ** -11                       # the lo step
NNZ = 7                              # non-zero entries per row at most: S(r) <= 7 (3/8 + E)^2 < 1
INT_MIN = -2 ** 31


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------------ grid data
def _entries(n, g):
    """n grid values: |a| = 1 (1/8 of them, b = 0) or |a| in {2, 3}; b = +-1 on 3/4 of the latter; random signs"""
    dev = g.device
    u = torch.randint(0, 8, (n,), generator=g, device=dev)
    mag = 1 + (u >= 1).long() + (u >= 5).long()
    v = torch.randint(0, 8, (n,), generator=g, device=dev)
    b = ((v >= 5).long() - ((v >= 2) & (v < 5)).long()) * (mag > 1).long()
    s = torch.randint(0, 2, (n,), generator=g, device=dev) * 2 - 1
    return (s.double() * mag.double() / 8 + b.double() * E).float()


def _sparse_rows(n, d, g, nnz=NNZ):
    """n rows with up to `nnz` grid entries at random columns"""
    dev = g.device
    M = torch.zeros(n, d, device=dev)
    cols = torch.randint(0, d, (n, nnz), generator=g, device=dev)
    M.scatter_(1, cols, _entries(n * nnz, g).view(n, nnz))
    return M


def _split(T, rz=False):
    """(hi, lo) of fp32 T as fp64: torch's round-to-nearest bf16 split, or round toward zero (truncation)"""
    T = T.float()
    if rz:
        hi = (T.view(torch.int32) & -65536).view(torch.float32)
        lo = ((T - hi).view(torch.int32) & -65536).view(torch.float32)
    else:
        hi = T.bfloat16().float()
        lo = (T - hi).bfloat16().float()
    return hi.double(), lo.double()


def _assert_on_grid(T, max_s=1.0):
    """The premise, on an actual tensor: hi + lo == T, hi = a / 8, lo = b / 2^11 with the rules above, S(row) <= max_s."""
    hi, lo = _split(T)
    assert torch.equal(hi + lo, T.double())
    a, b = hi * 8, lo / E
    assert torch.equal(a, a.round()) and float(a.abs().max()) <= 3
    assert torch.equal(b, b.round()) and float(b.abs().max()) <= 1
    assert not ((a.abs() == 1) & (b != 0)).any()
    assert float(((hi.abs() + lo.abs()) ** 2).sum(1).max()) <= max_s


def _rows_near(C, n, g, p_redraw=0.5, p_random=0.1):
    """n rows: a copy of a random centroid with each non-zero entry redrawn with probability p_redraw (same column, so
    x and its centroid overlap), or (p_random of them) a fresh sparse row.  Returns (X, source centroid of each row)."""
    dev = g.device
    k, d = C.shape
    src = torch.randint(0, k, (n,), generator=g, device=dev)
    X = C[src].clone()
    redraw = (torch.rand(n, d, generator=g, device=dev) < p_redraw) & (X != 0)
    X[redraw] = _entries(int(redraw.sum()), g)
    rnd = torch.rand(n, generator=g, device=dev) < p_random
    X[rnd] = _sparse_rows(int(rnd.sum()), d, g)
    return X, src


# Planted centroid pairs (p < q): identical except in one column j, where (c_p, c_q, x) are the values below (times a
# random sign); j is one of c_p's non-zero columns, and planted rows are x = c_p with column j set to x.
#   A  c_p = 2/8, c_q = 2/8 - E (same hi, lo -E), x = 2/8 - E: the formula picks p (x_lo . c_lo is left out), the true
#      distance q (x == c_q); without x_hi . c_lo, or with an RZ split of x or of c, the formula picks q.
#   B  c_p = 1/8, c_q = 3/8, x = 2/8 + E: x_lo . c_hi decides q; without it the two tie and p wins.
#   C  c_p = 2/8, c_q = 2/8 + E, x = 2/8: ||c_q||^2 - ||c_p||^2 = 2 (2/8) E + E^2 decides p; with ||c||^2 taken from the
#      hi plane the formula picks q.
#   D  c_q = c_p (lo planes not zero), x = c_p with its lo plane redrawn: lowest k wins, p.
PLANT = {'A': (2 / 8, 2 / 8 - E, 2 / 8 - E), 'B': (1 / 8, 3 / 8, 2 / 8 + E), 'C': (2 / 8, 2 / 8 + E, 2 / 8)}
FORMULA_PICKS_Q = {'A': False, 'B': True, 'C': False, 'D': False}
TRUTH_PICKS_Q = {'A': True, 'B': True, 'C': False, 'D': False}


def _plant(X, C, g):
    """Plant pairs at 31/32 (a 32-column chunk), 255/256 (a 256-column centroid tile), K-2/K-1 and a few low indices,
    kinds A, B, C, D in turn; about 10 % of the rows sit on them.  Returns [(kind, p, q, rows)]."""
    dev = g.device
    n, d = X.shape
    k = C.shape[0]
    pairs = []
    for p, q in ((31, 32), (255, 256), (k - 2, k - 1), (5, 6), (0, 9), (1, 3), (7, 8), (2, 4)):
        if 0 <= p < q < k and not {p, q} & {x for pq in pairs for x in pq}:
            pairs.append((p, q))
    rows = torch.randperm(n, generator=g, device=dev)
    per = n // (10 * len(pairs))
    out = []
    for i, (p, q) in enumerate(pairs):
        kind = 'ABCD'[i % 4]
        r = rows[i * per:(i + 1) * per]
        if kind == 'D':
            C[q] = C[p]
            hi, _ = _split(C[p])
            b = torch.randint(-1, 2, (len(r), d), generator=g, device=dev).double() * (hi.abs() >= 0.25)
            X[r] = (hi + b * E).float()
        else:
            nz = torch.nonzero(C[p]).view(-1)                   # a column c_p already uses: at most NNZ entries
            j = int(nz[torch.randint(0, len(nz), (1,), generator=g, device=dev)])
            s = float(torch.randint(0, 2, (1,), generator=g, device=dev)) * 2 - 1
            cp, cq, xv = PLANT[kind]
            C[p, j] = s * cp
            C[q] = C[p]
            C[q, j] = s * cq
            X[r] = C[p]
            X[r, j] = s * xv
        out.append((kind, p, q, r))
    return out


def _estep_data(n, d, k, g):
    C = _sparse_rows(k, d, g)
    X, src = _rows_near(C, n, g)
    plants = _plant(X, C, g)
    return X, C, src, plants


# ------------------------------------------------------------------------------------------------ fp64 references
def _formula(X, C, drop=(), rz_x=False, rz_c=False):
    """[N, K] fp64 distances of the E-step's documented form (not clamped: the kernel takes the argmin first and clamps
    only the row's minimum at 0, see _first_min).  Broken variants: drop any of
    'xl_ch', 'xh_cl' (a cross term), 'cn_lo', 'xn_lo' (the norm from the hi plane only); rz_x / rz_c: split by truncation."""
    xh, xl = _split(X, rz_x)
    ch, cl = _split(C, rz_c)
    Xd, Cd = X.double(), C.double()
    xn = (xh * xh).sum(1) if 'xn_lo' in drop else (Xd * Xd).sum(1)
    cn = (ch * ch).sum(1) if 'cn_lo' in drop else (Cd * Cd).sum(1)
    dot = xh @ ch.T
    if 'xh_cl' not in drop:
        dot += xh @ cl.T
    if 'xl_ch' not in drop:
        dot += xl @ ch.T
    return xn[:, None] + cn[None, :] - 2 * dot


def _true_dist(X, C):
    """[N, K] fp64 sum_d (x - c)^2, exact on the grid"""
    Xd, Cd = X.double(), C.double()
    return (Xd * Xd).sum(1)[:, None] + (Cd * Cd).sum(1)[None, :] - 2 * Xd @ Cd.T


def _first_min(dist):
    """(label = first minimum, minimum clamped at 0) per row, as the E-step kernels decide them"""
    m = dist.min(dim=1).values
    return (dist == m[:, None]).int().argmax(dim=1), m.clamp_min(0)


def _same(a, b):
    """equal values (-0 == +0), NaN exactly where the other has NaN"""
    a, b = a.double().cpu(), b.double().cpu()
    na, nb = a.isnan(), b.isnan()
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


def _check_plants(labels, plants, picks_q):
    for kind, p, q, rows in plants:
        want = q if picks_q[kind] else p
        assert (labels[rows] == want).all(), (kind, p, q, int((labels[rows] != want).sum()))


# Broken variants of the formula: (arguments, planted kind whose label it flips, least share of rows whose minimum
# distance it changes).  ||x||^2 is the same for every centroid of a row, so its variant moves distances, never labels.
# (Measured on this file's data at D = 40 .. 768, K = 12 .. 1000: 0.75-0.89 / 0.77-0.86 / 0.49-0.65 / 0.39-0.69 / 0.99-1.0 /
# 0.999-1.0 of the rows.)
VARIANTS = {
    'no x_lo.c_hi': (dict(drop=('xl_ch',)), 'B', 0.35),
    'no x_hi.c_lo': (dict(drop=('xh_cl',)), 'A', 0.35),
    'RZ split of x': (dict(rz_x=True), 'A', 0.25),
    'RZ split of c': (dict(rz_c=True), 'A', 0.2),
    '||c||^2 from hi': (dict(drop=('cn_lo',)), 'C', 0.5),
    '||x||^2 from hi': (dict(drop=('xn_lo',)), None, 0.5),
}


def _assert_every_part_is_seen(X, C, plants, want_m):
    for name, (kw, kind, share) in VARIANTS.items():
        lab, m = _first_min(_formula(X, C, **kw))
        changed = float((m != want_m).double().mean())
        assert changed >= share, (name, changed)
        if kind is not None:
            flip = {kd: (kd == kind) != FORMULA_PICKS_Q[kd] for kd in 'ABCD'}
            _check_plants(lab, [pl for pl in plants if pl[0] == kind], flip)


def test_split_grid_premise():
    """No GPU: the split identity and every bound of the module docstring hold on generated tensors (20 000 x 768 rows,
    7 non-zero entries per row, about two thirds of them with a lo part); hi.hi, hi.lo and lo.hi are non-zero against the
    row's centroid on most rows; the planted pairs decide as designed; and each broken variant of the formula changes the
    minimum distance on its share of the rows and the label on its planted rows."""
    g = torch.Generator().manual_seed(0)
    C = _sparse_rows(200, 768, g)
    X, src = _rows_near(C, 20000, g)
    for T in (X, C):
        _assert_on_grid(T)
    nz = X[X != 0]
    assert 0.6 < float((_split(nz)[1] != 0).double().mean()) < 0.72
    assert int((X != 0).sum(1).max()) == NNZ and NNZ * (3 / 8 + E) ** 2 < 1
    xh, xl = _split(X)
    ch, cl = _split(C[src])
    for a, b in ((xh, ch), (xh, cl), (xl, ch)):
        assert float(((a * b).sum(1) != 0).double().mean()) > 0.6
        assert torch.equal(a * b * 2 ** 14, (a * b * 2 ** 14).round())         # hi.hi on 2^-6, hi.lo on 2^-14
    assert torch.equal(X.double() ** 2 * 2 ** 22, (X.double() ** 2 * 2 ** 22).round())
    # 15 bits of accumulator, 24 bits of fma(-2, acc, ||c||^2), the final distance <= 2^24 units of 2^-22, fp64 inertia
    assert 3 * 2 ** 22 < 2 ** 24 and float(np.float32(4.0 - 2 ** -22)) == 4.0 - 2 ** -22
    assert (1 << 27) * 4 * 2 ** 22 < 2 ** 53
    # the M-step bound: sums below 2^13 on the 2^-11 grid are exact fp32
    assert float(np.float32(2 ** 13 - E)) == 2 ** 13 - E
    # the planted pairs and the sensitivity of each part, at a small shape
    g = torch.Generator().manual_seed(1)
    X, C, _, plants = _estep_data(4000, 72, 200, g)
    _assert_on_grid(X)
    _assert_on_grid(C)
    dist = _formula(X, C)
    want_l, want_m = _first_min(dist)
    _check_plants(want_l, plants, FORMULA_PICKS_Q)
    _check_plants(_first_min(_true_dist(X, C))[0], plants, TRUTH_PICKS_Q)
    _assert_every_part_is_seen(X, C, plants, want_m)


# ------------------------------------------------------------------------------------------------ E-step
def _run_estep(X, C, exact):
    labels = torch.empty(X.shape[0], dtype=torch.int64, device='cuda')
    mind = torch.empty(X.shape[0], dtype=torch.float32, device='cuda')
    acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    kmeans._estep(X, C, labels, acc, mind, exact=exact)
    return labels, mind, acc


def _assert_estep(labels, mind, acc, want_l, want_m):
    assert torch.equal(labels, want_l), int((labels != want_l).sum())
    assert torch.equal(mind.double(), want_m), int((mind.double() != want_m).sum())
    assert torch.equal(acc, want_m.sum().view(1))


@pytest.mark.gpu
@pytest.mark.parametrize('k,d', [(k, d) for d in (40, 72, 520, 768) for k in (12, 160, 161, 200, 257, 1000, 1024)])
def test_estep_equals_the_split_formula(k, d):
    """Tensor-core E-step (TMEM operand for K <= 160 at D >= 72, the ragged 16-column chunk at K = 161, several row tiles
    per CTA and 256-column centroid tiles for K > 256) against the documented formula: labels, distances and inertia equal
    on every row.  exact=True and pairwise_distance equal the TRUE distance instead, which differs on 44-80 % of the rows."""
    n = 148 * 128 * 2 + 77 if k > 256 else 6000 + k
    assert _lib.load().scd_estep_uses_tensor_cores(n, d, k) == 1
    g = torch.Generator(device='cuda').manual_seed(k * 1000 + d)
    X, C, _, plants = _estep_data(n, d, k, g)
    _assert_on_grid(X)
    _assert_on_grid(C)
    want_l, want_m = _first_min(_formula(X, C))
    _check_plants(want_l, plants, FORMULA_PICKS_Q)
    _assert_estep(*_run_estep(X, C, False), want_l, want_m)
    true = _true_dist(X, C)
    true_l, true_m = _first_min(true)
    _check_plants(true_l, plants, TRUTH_PICKS_Q)
    _assert_estep(*_run_estep(X, C, True), true_l, true_m)
    assert torch.equal(kmeans.pairwise_distance(X, C).double(), true)
    assert float((true_m != want_m).double().mean()) > 0.3                   # 2 x_lo . c_lo != 0: the two forms differ
    del true
    _assert_every_part_is_seen(X, C, plants, want_m)


# ------------------------------------------------------------------------------------------------ M-step
def _mstep_labels(n, k, g):
    """Clusters of 1, 31, 32 and 33 rows (they cross the segment sum's 32-row warp chunks), empty clusters first, in the
    middle and last, and labels -1 and K (ignored); small N: everything in the last cluster but one -1 and one K."""
    dev = g.device
    if n < 200:
        lab = torch.full((n,), k - 1, dtype=torch.int64, device=dev)
        if n > 2:
            lab[0], lab[1] = -1, k
    else:
        sizes = {0: 0, 1: 1, 2: 31, 3: 32, 4: 33, k // 2: 0, k - 1: 0}
        free = torch.tensor([c for c in range(k) if c not in sizes], device=dev)
        lab = free[torch.randint(0, len(free), (n,), generator=g, device=dev)]
        perm = torch.randperm(n, generator=g, device=dev)
        pos = 0
        for c, size in list(sizes.items()) + [(-1, n // 50), (k, n // 50)]:
            lab[perm[pos:pos + size]] = c
            pos += size
    return lab[torch.randperm(n, generator=g, device=dev)]


def _plane_bytes(k, d):
    return (k * d * 2 + 255) // 256 * 256


def _es_operands(es, k, d):
    """(hi, lo, ||c||^2) as the E-step workspace holds them"""
    pb = _plane_bytes(k, d)
    hi = es.ws[:k * d * 2].view(torch.bfloat16).view(k, d)
    lo = es.ws[pb:pb + k * d * 2].view(torch.bfloat16).view(k, d)
    return hi, lo, es.ws[2 * pb:2 * pb + 4 * k].view(torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize('n,d,k,aligned', [
    (1, 4, 1, True), (33, 100, 3, True), (127000, 128, 1000, True),           # segment_sum_kernel<2>, tail only / none
    (127000, 260, 11264, True),                                              # <2> with a tail, the sort's largest K
    (127000, 520, 100, True), (127000, 768, 1000, True),                     # <4> with a tail, <6>
    (127000, 1024, 100, True), (127000, 1148, 1000, True), (33, 1148, 1, True),   # <8>, <8> with the largest tail
    (33, 37, 3, True), (127000, 1152, 100, True), (127000, 768, 100, False),  # the generic kernel: D % 4, D > 1148, X % 16
])
def test_mstep_sums_and_centres_are_exact(n, d, k, aligned):
    """scd_mstep_sums: sums equal the fp64 group sums bit for bit (and two runs give the same bits), counts exact;
    finalize: centres == float32(sum / count), NaN rows for empty clusters, the same through counts_f; the E-step operands
    finalize(estep=...) leaves are torch's round-to-nearest split of those centres."""
    g = torch.Generator(device='cuda').manual_seed(n + d + k)
    dense = torch.rand(n, d, generator=g, device='cuda') < 0.5
    buf = torch.zeros(n * d + 1, device='cuda')
    X = buf[int(not aligned):int(not aligned) + n * d].view(n, d)
    X[dense] = _entries(int(dense.sum()), g)
    assert (X.data_ptr() % 16 == 0) == aligned
    _assert_on_grid(X, max_s=d)
    labels = _mstep_labels(n, k, g)
    ok = (labels >= 0) & (labels < k)
    want_s = torch.zeros(k, d, dtype=torch.float64, device='cuda').index_add_(0, labels[ok], X[ok].double())
    bound = torch.zeros(k, d, dtype=torch.float64, device='cuda').index_add_(0, labels[ok], X[ok].double().abs())
    assert float(bound.max()) < 2 ** 13                                      # exact in fp32 in any order
    want_c = torch.bincount(labels[ok], minlength=k)
    assert n < 200 or all(int(want_c[c]) == s for c, s in ((0, 0), (1, 1), (2, 31), (3, 32), (4, 33), (k // 2, 0), (k - 1, 0)))
    ms = kmeans._MStep(n, d, k, 'cuda')
    ms.sums_counts(X, labels)
    sums1 = ms.sums.clone()
    assert torch.equal(sums1.double(), want_s), int((sums1.double() != want_s).sum())
    assert torch.equal(ms.counts.long(), want_c)
    ms.sums_counts(X, labels)
    assert torch.equal(ms.sums.view(torch.int32), sums1.view(torch.int32))
    want = (want_s / want_c.double()[:, None]).float()                       # double rounding is harmless for '/'
    es = kmeans._EStep(k, d, 'cuda')
    got = torch.empty(k, d, device='cuda')
    ms.finalize(None, got, estep=es)
    assert _same(got, want)
    assert torch.isnan(got[want_c == 0]).all() and not torch.isnan(got[want_c > 0]).any()
    got_f = torch.full((k, d), 7.0, device='cuda')
    ms.finalize(None, got_f, counts_f=ms.counts.float())
    assert _same(got_f, want)
    hi, lo, _ = _es_operands(es, k, d)
    assert _same(hi.float(), want.bfloat16().float())
    assert _same(lo.float(), (want - want.bfloat16().float()).bfloat16().float())


# ------------------------------------------------------------------------------------------------ the loop's chain
@pytest.mark.gpu
@pytest.mark.parametrize('k,d', [(12, 40), (161, 768), (257, 72), (1000, 520), (1024, 768)])
def test_mstep_finalize_then_estep_on_the_grid(k, d):
    """Clusters of a grid centre plus symmetric pairs c +- delta (and sometimes c itself) have the centre as their exact
    mean: sums_counts -> finalize(estep=...) gives the centres bit for bit and leaves torch's split of them and their exact
    ||c||^2 in the E-step workspace; the E-step on fresh grid rows with SCD_ESTEP_PLANES_READY then equals the formula and
    the launch that splits the centres itself."""
    g = torch.Generator(device='cuda').manual_seed(k + d)
    C = _sparse_rows(k, d, g, nnz=NNZ - 1)                                   # room for delta's one column
    npairs = torch.randint(1, 13, (k,), generator=g, device='cuda')
    owner = torch.repeat_interleave(torch.arange(k, device='cuda'), npairs)
    m = owner.numel()
    j = torch.randint(0, d, (m,), generator=g, device='cuda')
    v = C[owner, j]
    hv, lv = _split(v)
    delta = torch.where(v == 0, _entries(m, g), torch.where((lv == 0) & (hv.abs() >= 0.25), E, 0.0).float())
    plus, minus = C[owner].clone(), C[owner].clone()
    plus[torch.arange(m), j] += delta
    minus[torch.arange(m), j] -= delta
    single = torch.nonzero(torch.rand(k, generator=g, device='cuda') < 0.5).view(-1)
    Xfit = torch.cat((plus, minus, C[single]))
    lab = torch.cat((owner, owner, single))
    perm = torch.randperm(Xfit.shape[0], generator=g, device='cuda')
    Xfit, lab = Xfit[perm].contiguous(), lab[perm].contiguous()
    _assert_on_grid(Xfit)
    assert float((delta != 0).double().mean()) > 0.5
    ms, es = kmeans._MStep(Xfit.shape[0], d, k, 'cuda'), kmeans._EStep(k, d, 'cuda')
    ms.sums_counts(Xfit, lab)
    c_new = torch.empty(k, d, device='cuda')
    ms.finalize(None, c_new, estep=es)
    assert torch.equal(c_new, C)
    hi, lo, cn = _es_operands(es, k, d)
    ch, cl = _split(C)
    assert torch.equal(hi.double(), ch) and torch.equal(lo.double(), cl) and bool((cl != 0).any())
    assert torch.equal(cn.double(), (C.double() ** 2).sum(1))
    X, _ = _rows_near(C, 148 * 128 + 5, g)
    want_l, want_m = _first_min(_formula(X, C))
    got = torch.empty(X.shape[0], dtype=torch.int64, device='cuda'), torch.empty(X.shape[0], device='cuda')
    acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    assert es.ready_for == c_new.data_ptr()
    es.run(X, c_new, got[0], acc, got[1])                                   # the operands finalize left behind
    _assert_estep(*got, acc, want_l, want_m)
    _assert_estep(*_run_estep(X, c_new, False), want_l, want_m)             # centroid_split_kernel's own


# ------------------------------------------------------------------------------------------------ labelled inertia
@pytest.mark.gpu
@pytest.mark.parametrize('n,d', [(1, 768), (5, 40), (7, 20), (300, 37), (127000, 768)])
def test_labelled_inertia_is_exact(n, d):
    """scd_labelled_inertia (one warp per row, fp64 atomics per block) equals the fp64 sum of ||l_i - c_label||^2 over
    the rows with a label in [0, K): fewer rows than the block's 8 warps, D below and above the 32 lanes, large N."""
    k = 100
    g = torch.Generator(device='cuda').manual_seed(n + d)
    C = _sparse_rows(k, d, g)
    L, src = _rows_near(C, n, g)
    labels = src.clone()
    if n > 2:
        labels[torch.randperm(n, generator=g, device='cuda')[:max(1, n // 20)]] = -1
        labels[torch.randperm(n, generator=g, device='cuda')[:max(1, n // 20)]] = k
    _assert_on_grid(L)
    ok = (labels >= 0) & (labels < k)
    want = ((L[ok].double() - C[labels[ok]].double()) ** 2).sum()
    acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    lib = _lib.load()
    _lib.check(lib.scd_labelled_inertia(L.data_ptr(), labels.data_ptr(), n, d, C.data_ptr(), k, acc.data_ptr(), _stream()),
               'scd_labelled_inertia')
    assert torch.equal(acc, want.view(1))


# ------------------------------------------------------------------------------------------------ k-means++
@pytest.mark.gpu
def test_kpp_update_is_exact():
    """scd_kpp_update on grid rows: d2 (the first step assigns, later steps take the min), the per-64-row fp64 block sums
    in the workspace and center_out are exact; the center= form (the row-sharded seeding) gives the same bits."""
    lib = _lib.load()
    n, d = 20000 + 37, 100
    g = torch.Generator(device='cuda').manual_seed(3)
    C = _sparse_rows(40, d, g)
    X, _ = _rows_near(C, n, g)
    _assert_on_grid(X)
    nb = (n + 63) // 64
    ws = torch.zeros(lib.scd_kpp_workspace_bytes(n), dtype=torch.uint8, device='cuda')
    ws2 = torch.zeros_like(ws)
    d2, d2b = torch.full((n,), -1.0, device='cuda'), torch.full((n,), -1.0, device='cuda')
    centre = torch.empty(d, device='cuda')
    want = None
    for step, idx in enumerate([5, n - 1, 64, 1234, 63]):
        pick = torch.tensor([idx], dtype=torch.int64, device='cuda')
        _lib.check(lib.scd_kpp_update(X.data_ptr(), n, d, pick.data_ptr(), None, int(step == 0), d2.data_ptr(), centre.data_ptr(),
                                      ws.data_ptr(), ws.numel(), _stream()), 'scd_kpp_update')
        _lib.check(lib.scd_kpp_update(X.data_ptr(), n, d, None, X[idx].contiguous().data_ptr(), int(step == 0), d2b.data_ptr(), None,
                                      ws2.data_ptr(), ws2.numel(), _stream()), 'scd_kpp_update')
        dist = ((X.double() - X[idx].double()) ** 2).sum(1)
        want = dist if want is None else torch.minimum(want, dist)
        assert torch.equal(d2.double(), want) and torch.equal(centre, X[idx])
        sums = torch.zeros(nb * 64, dtype=torch.float64, device='cuda')
        sums[:n] = want
        assert torch.equal(ws[:nb * 8].view(torch.float64), sums.view(nb, 64).sum(1))
        assert torch.equal(d2b, d2) and torch.equal(ws2[:nb * 8], ws[:nb * 8])


def _kpp_select(d2, r):
    lib = _lib.load()
    n = d2.numel()
    ws = torch.empty(lib.scd_kpp_workspace_bytes(n), dtype=torch.uint8, device='cuda')
    pick = torch.full((1,), -1, dtype=torch.int64, device='cuda')
    no_hit = torch.zeros(1, dtype=torch.int32, device='cuda')
    _lib.check(lib.scd_kpp_select(d2.data_ptr(), n, 0, float(r), pick.data_ptr(), no_hit.data_ptr(), ws.data_ptr(), ws.numel(),
                                  _stream()), 'scd_kpp_select')
    assert int(no_hit.item()) == 0
    return int(pick.item())


@pytest.mark.gpu
def test_kpp_select_pins_the_first_row_reaching_the_draw():
    """scd_kpp_select on d2 in multiples of 2^-10 with a power-of-two total, so r = cum[i] / total and r * total are exact:
    r == cum[i] / total picks i; nextafter(r, 1) picks the next row with a non-zero d2, skipping zero rows and crossing
    64-row block edges; r = 0 picks row 0, also when d2[0] == 0."""
    n = 300
    g = torch.Generator().manual_seed(11)
    for zeros, cases in (
        ([1, 62, 64, 65, 66, 128, n - 2], {0: 2, 63: 67, 127: 129, n - 3: n - 1, n - 1: n - 1, 100: 101}),
        ([0, 63, 200], {62: 64, 64: 65, 199: 201, 191: 192}),
    ):
        units = torch.randint(1, 9, (n,), generator=g).double()
        units[zeros] = 0
        units[150] += 2.0 ** int(np.ceil(np.log2(float(units.sum())))) - float(units.sum())     # total: a power of two
        d2 = units / 1024
        cum = torch.cumsum(d2, 0).numpy()
        total = float(cum[-1])
        assert total == 2.0 ** round(np.log2(total)) and torch.equal(d2.float().double(), d2)
        d2c = d2.float().cuda()
        for i, nxt in cases.items():
            assert d2[i] > 0
            r = float(cum[i]) / total
            assert r * total == cum[i]
            assert _kpp_select(d2c, r) == i == int(np.searchsorted(cum, r * total, side='left'))
            r1 = float(np.nextafter(r, 1.0))
            assert _kpp_select(d2c, r1) == nxt == min(int(np.searchsorted(cum, r1 * total, side='left')), n - 1)
        assert _kpp_select(d2c, 0.0) == 0
    assert d2[0] == 0                                                        # the second d2 starts with a zero row


# ------------------------------------------------------------------------------------------------ int32 costs
@pytest.mark.gpu
def test_cost_x1000_on_the_grid():
    """constrained_int_costs == np.around(float64(float32 sqrt(d)) * 1000) on exact distances, NaN (an empty cluster's
    centre) -> INT_MIN."""
    g = torch.Generator(device='cuda').manual_seed(5)
    C = _sparse_rows(70, 72, g)
    X, _ = _rows_near(C, 3000, g)
    C[[0, 69]] = float('nan')
    d = _true_dist(X, C).float().cpu().numpy()
    d[:, [0, 69]] = np.nan
    with np.errstate(invalid='ignore'):
        want = np.around(np.sqrt(d).astype(np.float64) * 1000)
    want = np.where(np.isnan(want), INT_MIN, want).astype(np.int64)
    got = kmeans.constrained_int_costs(X, C).cpu().numpy()
    assert got.dtype == np.int32 and np.array_equal(got.astype(np.int64), want)
    assert (np.isnan(d) == (got == INT_MIN)).all()
