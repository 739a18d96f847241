"""GPU: the scoring kernel's vocabulary ring of 32-k half k-blocks and its warp roles.

A k-block's first two MMAs read one vocabulary stage and its last two the next, so a ragged last k-block has a half
that lies partly or wholly beyond D (TMA fills it with zeros).  Widths D <= 128 have fewer k-blocks per tile than MMA
issuers and take the waits after the issue token.  Large row counts give a CTA pair several work items, and ranges that
end in one-tile items.  Every case is checked against the oracle on a row sample, and a second launch must equal the
first bit for bit.
"""
import pytest
import torch

from oracle import naming_oracle
from scd_b200 import naming

pytestmark = pytest.mark.gpu
TAU = 1e-3
LOGIT_ATOL = 2e-3
SOFTMAX_ATOL = 1e-5


def _check_against_oracle(vals, idx, X, W, k, softmax):
    """X: [n, d] float rows, W: [d, v] float.  Values within the tolerance of the oracle; indices equal wherever the
    logit gaps to both neighbours (the (k+1)-th score included) exceed TAU."""
    variant = 'unsup' if softmax else 'ptsup'
    kk = min(k, W.shape[1])
    oi, ov = naming_oracle.score_topk(X, W, min(k + 1, W.shape[1]), variant=variant)
    vals, idx = vals.cpu()[:, :kk], idx.cpu()[:, :kk]
    atol = SOFTMAX_ATOL if softmax else LOGIT_ATOL
    assert torch.allclose(vals, ov[:, :kk], atol=atol, rtol=0), float((vals - ov[:, :kk]).abs().max())
    lv = ov if not softmax else naming_oracle.score_topk(X, W, min(k + 1, W.shape[1]), variant='ptsup')[1]
    n = len(X)
    gaps = lv[:, :-1] - lv[:, 1:] if lv.shape[1] > 1 else torch.full((n, 0), 1e9)
    if lv.shape[1] == kk:
        gaps = torch.cat((gaps, torch.full((n, 1), 1e9)), dim=1)
    clear = gaps > TAU
    left = torch.cat((torch.ones(n, 1, dtype=torch.bool), clear[:, :kk - 1]), dim=1)
    pinned = left & clear[:, :kk]
    assert pinned.float().mean() > 0.97
    assert torch.equal(idx[pinned], oi[:, :kk][pinned])


def _run_and_check(n, v, d, k, softmax, sample):
    g = torch.Generator().manual_seed(n + 7 * v + 13 * d + k)
    X = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).bfloat16()
    W = torch.nn.functional.normalize(torch.randn(v, d, generator=g), dim=1).bfloat16()
    Xc = X.cuda()
    vocab = naming.Vocabulary.from_rows(W.cuda())
    v0, i0, m0, s0 = naming.name_topk_raw(Xc, vocab, k, softmax, want_stats=softmax)
    v0, i0 = v0.clone(), i0.clone()
    v1, i1, m1, s1 = naming.name_topk_raw(Xc, vocab, k, softmax, want_stats=softmax)
    assert torch.equal(v0, v1) and torch.equal(i0, i1)
    if softmax:
        assert torch.equal(m0, m1) and torch.equal(s0, s1)
    rows = torch.randperm(n, generator=g)[:sample] if sample < n else torch.arange(n)
    _check_against_oracle(v0[rows.cuda()], i0[rows.cuda()], X[rows].float(), W.float().t().contiguous(), k, softmax)


@pytest.mark.parametrize('softmax', [False, True])
@pytest.mark.parametrize('k', [1, 5, 8])
@pytest.mark.parametrize('d', [72, 96, 200, 520])
def test_ragged_last_half_k_block(d, k, softmax):
    """D = 72 / 96: the second half of the last k-block is wholly beyond D (and D <= 128: post-token waits);
    D = 200 / 520: the last k-block's first half is ragged and its second half empty."""
    _run_and_check(3000, 2500, d, k, softmax, sample=3000)


@pytest.mark.parametrize('n,v,d,k,softmax', [(19000, 5000, 96, 5, False), (19000, 5000, 200, 8, True),
                                             (40000, 11000, 72, 5, False), (30000, 3000, 520, 1, True),
                                             (19000, 5000, 128, 1, False), (60000, 2000, 768, 8, False)])
def test_multi_item_and_one_tile_item_shapes(n, v, d, k, softmax):
    """Several work items per CTA pair and one-tile items at range ends, through the split vocabulary ring."""
    _run_and_check(n, v, d, k, softmax, sample=1500)
