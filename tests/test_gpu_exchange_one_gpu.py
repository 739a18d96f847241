"""The peer-memory exchange kernels on ONE GPU with simulated ranks: record packing (scd_pack_vote_records_peer,
scd_pack_sorted_records_peer), the segmented vote (scd_vote_segments), the fused all-reduce + divide of the M-step
(scd_finalize_centers_peer), the flag protocol of scd_peer_barrier and a CUDA graph replaying the device-side epochs.

All of these kernels take plain device pointers: a table of G buffer bases that double as the G flag pads.  Here G ordinary
allocations stand in for the G mapped buffers, laid out by the product's own ``PeerExchange._carve``; a store "to rank r"
is a local store and the rank-ordered peer loads are local loads.  Virtual ranks launch one after another on one stream.
What this cannot show - NVLink memory ordering, the symmetric-memory mapping, the timeout trap - stays with
test_gpu_peer.py.

Barrier rule: a launch never waits.  Before every launch that contains a barrier, ``Ranks.launch`` raises the arrive words
of the other ranks on the launching rank's pad to the epoch the barrier is going to wait for and checks on the host that
the wait condition holds, so a mistake in this file fails in Python instead of spinning on the GPU."""

import numpy as np
import pytest
import torch

from oracle import naming_oracle
from scd_b200 import _lib, dist as sdist, kmeans, naming, peer, synth
from test_gpu_kmeans_split_grid import _assert_on_grid, _rows_near, _sparse_rows

pytestmark = pytest.mark.gpu

# Flag pad of a rank (peer_kernel.cuh:15-19, 28-31): 8 channels of 32 words, channel c = arrive[16] | epoch | ticket | pad
CHANNELS, CH_WORDS, EPOCH, TICKET = 8, 32, 16, 17
SENTINEL = 0xA5
SLACK = 4096                       # bytes after the layout: stray stores past the last record array stay in the allocation
M = 20                             # names voted per cluster


class _VirtualRank(peer.PeerExchange):
    """A ``PeerExchange`` whose buffers are ordinary allocations of one GPU (no process group, no symmetric memory)."""

    def __init__(self, bufs, rank, k, d, n_total, k_used):
        self._carve(len(bufs), rank, k, d, n_total, k_used, bufs[rank], [b.data_ptr() for b in bufs])


class Ranks:
    """G virtual ranks over G buffers: zero flag pads, everything else SENTINEL."""

    def __init__(self, world, k, d, n_total=0, k_used=0):
        # Ranks.launch addresses flag words through this layout: a pad of another size fails here, before any launch
        assert _lib.load().scd_peer_flag_bytes() == CHANNELS * CH_WORDS * 4
        nbytes = peer.PeerExchange.buffer_bytes(world, k, d, n_total, k_used)
        self.bufs = [torch.full((nbytes + SLACK,), SENTINEL, dtype=torch.uint8, device='cuda') for _ in range(world)]
        self.px = [_VirtualRank(self.bufs, r, k, d, n_total, k_used) for r in range(world)]
        self.flag_bytes = self.px[0].off_mstep
        for b in self.bufs:
            b[:self.flag_bytes].zero_()
        self.world = world
        self.done = np.zeros((world, CHANNELS), dtype=np.int64)    # barrier launches per (rank, channel)

    def pad(self, r):
        return self.bufs[r][:CHANNELS * CH_WORDS * 4].view(torch.int32).view(CHANNELS, CH_WORDS)

    def pads(self):
        torch.cuda.synchronize()
        return np.stack([self.pad(r).cpu().numpy().astype(np.int64) for r in range(self.world)])

    def launch(self, rank, channel, fn):
        """``fn()`` launches exactly one barrier of virtual rank ``rank`` on ``channel`` (and any number of launches without
        one); run it only once that barrier's wait condition already holds, then check the flag protocol."""
        G = self.world
        pads = self.pads()
        epoch = int(pads[rank, channel, EPOCH])
        assert epoch == self.done[rank, channel], (rank, channel, epoch)
        target = epoch + 1
        pad = self.pad(rank)
        for q in range(G):
            if q != rank:
                pad[channel, q] = max(int(pads[rank, channel, q]), target)
        before = self.pads()
        assert all(before[rank, channel, q] >= target for q in range(G) if q != rank)    # the barrier cannot wait
        out = fn()
        after = self.pads()
        self.done[rank, channel] += 1
        assert after[rank, channel, EPOCH] == target
        assert after[rank, channel, TICKET] == 0
        assert all(after[q, channel, rank] == target for q in range(G))
        want = before.copy()
        want[:, channel, rank] = target
        want[rank, channel, EPOCH] = target
        assert np.array_equal(after, want)                    # nothing else moved, other channels included
        return out


# ------------------------------------------------------------------------------------------------ references
def _vote_ref(idx, labels, K, k_used, known=None):
    """vote_device on the unsharded arrays (host copies)"""
    out = naming.vote_device(idx.cuda(), labels.cuda(), K, k_used, M, known_name_idx=known)
    assert int(out[4].item()) == 0
    return [t.cpu() for t in out[:4]]


def _assert_vote(got, want, idx, labels, K, k_used, known=None):
    names, counts, distinct, rows, ovf = got
    assert int(ovf.item()) == 0
    for a, b in zip((names, counts, distinct, rows), want):
        assert torch.equal(a.cpu(), b)
    # Counter.most_common on the largest cluster, an empty one and a few others
    sizes = torch.bincount(labels, minlength=K)
    sample = {int(sizes.argmax()), int(sizes.argmin()), 0, K - 1, K // 2}
    assert int(sizes.min()) == 0
    co = naming_oracle.vote(idx, labels.numpy(), sorted(sample), k_used, known_name_idx=known)
    for c in sample:
        want_c = [(int(a), int(b)) for a, b in co[c].most_common(M)]
        assert [(int(a), int(b)) for a, b in zip(want[0][c].tolist(), want[1][c].tolist()) if a >= 0] == want_c, c


def _names(n, k_total, v, g):
    """top-k lists with a heavy head (many equal counts per cluster)"""
    return (torch.rand(n, k_total, generator=g) ** 4 * v).long()


# ------------------------------------------------------------------------------------------------ A: unsorted records
@pytest.mark.parametrize('misaligned', [False, True])
@pytest.mark.parametrize('k_used', [1, 2, 4, 5, 8])
@pytest.mark.parametrize('world', [2, 3, 7, 16])
def test_pack_vote_records_peer_then_vote_records(world, k_used, misaligned):
    """Every buffer holds [label, names[:k_used]] of every row, nothing outside that range is written, and the vote on each
    buffer equals the unsharded vote.  n_total = 613 G - 1: three tiles per shard (the last one odd), odd `per` (odd ranks
    start on an odd word when 1 + k_used is odd) and a ragged last shard.  misaligned: the records start 4 bytes after
    the layout's 256-aligned offset, so every tile takes the 4-byte stores."""
    g = torch.Generator().manual_seed(world * 100 + k_used)
    n, K, k_total = 613 * world - 1, 37, 8
    labels = torch.randint(0, K - 1, (n,), generator=g)            # cluster K - 1 stays empty
    labels[:700] = 3                                               # a large cluster across the first shards
    idx = _names(n, k_total, 400, g)
    rk = Ranks(world, K, 8, n_total=n, k_used=k_used)
    per, w = rk.px[0].per, 1 + k_used
    assert per == 613 and n % world
    rec_base = rk.px[0]._records[0][1] + (4 if misaligned else 0)
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    for r in range(world):
        lo, hi = sdist.shard_bounds(n, world, r)
        lab_r, idx_r = labels[lo:hi].cuda(), idx[lo:hi].cuda()
        if misaligned:                                             # no barrier: nothing waits
            _lib.check(lib.scd_pack_vote_records_peer(rk.px[r].table, world, r, rec_base, lab_r.data_ptr(), idx_r.data_ptr(),
                                                      k_total, k_used, hi - lo, r * per, st), 'scd_pack_vote_records_peer')
        else:
            rk.launch(r, peer.RECORD_CHANNEL, lambda: rk.px[r].gather_records(lab_r, idx_r, k_used))
    torch.cuda.synchronize()
    want_rec = torch.cat((labels[:, None], idx[:, :k_used]), 1).int()
    want = _vote_ref(idx, labels, K, k_used)
    end = rec_base + n * w * 4
    for r in range(world):
        b = rk.bufs[r]
        rec = b[rec_base:end].view(torch.int32).view(n, w)
        assert torch.equal(rec.cpu(), want_rec)
        assert bool((b[rk.flag_bytes:rec_base] == SENTINEL).all()) and bool((b[end:] == SENTINEL).all())
        got = naming.vote_records(rec, K, M)
        _assert_vote(got, want, idx, labels, K, k_used)


# ------------------------------------------------------------------------------------------------ B: sorted runs
def _sorted_case(case, g):
    """(world, n, K, k_used, labels, idx, known): clusters spread over all ranks, clusters that live on one rank (labels
    follow the row id), empty clusters, and a small vocabulary so counts tie a lot"""
    world, n, K, k_used, big = case
    labels = torch.randint(0, K // 2, (n,), generator=g) * 2        # even clusters: spread (and some left empty)
    per = (n + world - 1) // world
    for r in range(world):                                         # odd clusters: one block of rows inside one shard
        lo, hi = sdist.shard_bounds(n, world, r)
        c = 1 + 2 * (r % max(1, K // 2 - 1))
        labels[lo + per // 4:lo + per // 4 + min(per // 3, 50)][:max(0, hi - lo - per // 4)] = c
    labels[labels == K - 2] = 0                                     # clusters K - 2 and K - 1 stay empty
    idx = _names(n, 8, 60, g)
    if big:                                                         # two clusters of > 8192 entries each, > 16384 names each
        sel = torch.rand(n, generator=g) < 0.8
        labels[sel] = torch.randint(0, 2, (int(sel.sum()),), generator=g) * 2
        idx[sel] = torch.randint(0, 90_000, (int(sel.sum()), 8), generator=g)
    known = [int(x) for x in idx[:40, 0].unique()[:5]]
    return world, n, K, k_used, labels, idx, known


def _reverse_runs(rec, seg, per):
    """the same records with every (rank, cluster) run reversed - another valid label-sorted order"""
    out = rec.clone()
    seg_h = seg.cpu()
    for r in range(seg_h.shape[0]):
        for c in range(seg_h.shape[1] - 1):
            a, b = r * per + int(seg_h[r, c]), r * per + int(seg_h[r, c + 1])
            if b - a > 1:
                out[a:b] = rec[a:b].flip(0)
    return out


B_CASES = {'g2_k5': (2, 3001, 40, 5, False), 'g5_k1': (5, 4099, 40, 1, False), 'g16_k8': (16, 5003, 40, 8, False),
           'g16_empty_shards': (16, 20, 8, 5, False), 'g5_spill_k5': (5, 50_001, 6, 5, True),
           'g16_spill_k1': (16, 40_003, 6, 1, True)}


@pytest.mark.parametrize('case', list(B_CASES))
def test_pack_sorted_records_peer_then_vote_segments(case):
    """Each virtual rank sorts its shard with its own _MStep (not a stable sort) and stores its runs + offsets into every
    buffer; the offsets tables, unpack_sorted and vote_segments (also with excluded names, and on runs in reversed order,
    where first occurrences must come from the row ids) equal the unsharded arrays and vote."""
    g = torch.Generator().manual_seed(len(case) * 7 + B_CASES[case][1])
    world, n, K, k_used, labels, idx, known = _sorted_case(B_CASES[case], g)
    rk = Ranks(world, K, 4, n_total=n, k_used=k_used)
    per = rk.px[0].per
    shards = [sdist.shard_bounds(n, world, r) for r in range(world)]
    if case == 'g16_empty_shards':
        assert shards[-1][0] == shards[-1][1] == n
    out = []
    for r, (lo, hi) in enumerate(shards):
        ms = kmeans._MStep(hi - lo, 4, K, 'cuda')
        ms.sums_counts(torch.randn(hi - lo, 4, generator=g).cuda(), labels[lo:hi].cuda())
        idx_r = idx[lo:hi].cuda()
        out.append(rk.launch(r, peer.RECORD_CHANNEL, lambda: rk.px[r].gather_sorted_records(ms, idx_r, k_used)))
    torch.cuda.synchronize()
    offs = torch.stack([torch.cat((torch.zeros(1, dtype=torch.long),
                                   torch.bincount(labels[lo:hi], minlength=K).cumsum(0))) for lo, hi in shards]).int()
    want = _vote_ref(idx, labels, K, k_used)
    want_x = _vote_ref(idx, labels, K, k_used, known)
    px0 = rk.px[0]
    rec_end = px0.off_rec + n * (1 + k_used) * 4
    seg_end = px0.off_seg + world * (K + 1) * 4
    for r in range(world):
        rec, seg = out[r]
        b = rk.bufs[r]
        # nothing stored outside the parity-0 records and offsets table: M-step blocks, parity-1 arrays, slack
        for lo, hi in ((rk.flag_bytes, px0.off_rec), (rec_end, px0.off_seg), (seg_end, b.numel())):
            assert bool((b[lo:hi] == SENTINEL).all()), (lo, hi)
        assert torch.equal(seg.cpu(), offs)
        lab_u, idx_u = rk.px[r].unpack_sorted(rec, seg)
        assert torch.equal(lab_u.cpu(), labels) and torch.equal(idx_u.cpu(), idx[:, :k_used])
        got = naming.vote_segments(rec, seg, K, M, n_total=n)
        _assert_vote(got, want, idx, labels, K, k_used)
        if B_CASES[case][4] and k_used == 5:
            assert int(got[2][0]) > 16384 and int(got[2][2]) > 16384                 # the spill tables of vote_kernel<SEG>
        got = naming.vote_segments(rec, seg, K, M, known_name_idx=known, n_total=n)
        _assert_vote(got, want_x, idx, labels, K, k_used, known)
    got = naming.vote_segments(_reverse_runs(out[0][0], out[0][1], per), out[0][1], K, M, n_total=n)
    _assert_vote(got, want, idx, labels, K, k_used)


# ------------------------------------------------------------------------------------------------ C: finalize_centers_peer
def _mstep_blocks(world, K, D, g):
    """per-rank (sums fp32 [K, D], counts int32 [K], inertia fp64): clusters empty on every rank (NaN rows) and clusters
    counted on one rank only; a rank's sums are zero where its count is"""
    counts = torch.randint(1, 50, (world, K), generator=g, dtype=torch.int32)
    counts[:, torch.arange(K) % 7 == 3] = 0
    one = torch.arange(K) % 5 == 1
    counts[:, one] = 0
    counts[torch.randint(0, world, (int(one.sum()),), generator=g), one.nonzero().view(-1)] = 17
    sums = torch.randn(world, K, D, generator=g) * counts[:, :, None].float()
    sums[counts == 0] = 0
    inertia = torch.rand(world, generator=g, dtype=torch.float64) * 1e4
    return sums, counts, inertia


def _finalize_ref(sums, counts, inertia):
    """float32 adds in rank order from 0.f, IEEE divide; fp64 inertia in rank order"""
    s = np.zeros(sums.shape[1:], dtype=np.float32)
    for r in range(sums.shape[0]):
        s = s + sums[r].numpy()
    cnt = counts.long().sum(0).numpy().astype(np.float32)
    with np.errstate(invalid='ignore', divide='ignore'):
        c = s / cnt[:, None]
    t = 0.0
    for r in range(inertia.shape[0]):
        t += float(inertia[r])
    return torch.from_numpy(s), torch.from_numpy(c), torch.from_numpy(cnt), t


def _bits_equal(a, b):
    """bit-equal, NaN exactly where the other has NaN (NaN payloads may differ between the host and the device)"""
    a, b = a.cpu(), b.cpu()
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na].view(torch.int32), b[~nb].view(torch.int32))


def _es_planes(ws, k, d):
    """(hi plane, lo plane, ||c||^2) bytes of an E-step workspace"""
    pb = (k * d * 2 + 255) // 256 * 256
    return ws[:k * d * 2], ws[pb:pb + k * d * 2], ws[2 * pb:2 * pb + 4 * k]


def _bytes(t):
    return t if t.dtype == torch.uint8 else t.view(torch.uint8)


def _run_finalize(rk, world, K, D, parity, c_old):
    outs = []
    for r in range(world):
        px = rk.px[r]
        block = px._blocks[parity]
        c_new = torch.full((K, D), 7.0, device='cuda')
        norms = torch.full((K,), -1.0, device='cuda')
        cnt = torch.full((K,), -1.0, device='cuda')
        inert = torch.full((1,), -1.0, dtype=torch.float64, device='cuda')
        es = kmeans._EStep(K, D, 'cuda')
        es.ws.zero_()
        rk.launch(r, peer.MSTEP_CHANNEL, lambda: px.finalize(block, c_old, c_new, norms, cnt, inert, es))
        outs.append((c_new, norms, cnt, inert, es))
    return outs


@pytest.mark.parametrize('k,d', [(1, 8), (100, 768), (1000, 512), (37, 6), (5, 129)])
@pytest.mark.parametrize('world', [2, 3, 8, 16])
def test_finalize_centers_peer_is_the_rank_order_sum(world, k, d):
    """Centres, counts and inertia equal an exact host reference bit for bit; the next E-step's operands equal the local
    scd_finalize_centers' on the rank-summed buffer byte for byte (and torch's split of the centres); every virtual rank
    gets the same bits, from both parity blocks; null optional outputs are accepted.  K = 1000 is more blocks than SMs;
    D = 6 and 129 take the scalar peer loads, and 37 * 6 + 37 is odd (the inertia's pad word)."""
    g = torch.Generator().manual_seed(world * 10_000 + k + d)
    rk = Ranks(world, k, d)
    c_old = torch.randn(k, d, generator=g).cuda()
    for parity in (0, 1):
        sums, counts, inertia = _mstep_blocks(world, k, d, g)
        for r in range(world):
            blk = rk.px[r].next_mstep_block()
            assert blk[3] == rk.px[r]._blocks[parity][3] > 0
            blk[0].copy_(sums[r])
            blk[1].copy_(counts[r])
            blk[2].fill_(float(inertia[r]))
        s_ref, c_ref, cnt_ref, t_ref = _finalize_ref(sums, counts, inertia)
        outs = _run_finalize(rk, world, k, d, parity, c_old)
        c_new, norms, cnt, inert, es = outs[0]
        assert _bits_equal(c_new, c_ref)
        assert torch.equal(torch.isnan(c_new).all(1).cpu(), counts.sum(0) == 0) and not torch.isnan(c_new[counts.sum(0) > 0]).any()
        assert torch.equal(cnt.cpu(), cnt_ref)
        assert float(inert) == t_ref
        ref_n = ((c_ref.double() - c_old.cpu().double()) ** 2).sum(1).sqrt()
        assert torch.equal(torch.isnan(norms.cpu()), torch.isnan(ref_n))
        ok = ~torch.isnan(ref_n)
        assert torch.allclose(norms.cpu()[ok].double(), ref_n[ok], rtol=1e-6, atol=0)
        for o in outs[1:]:                                              # identical bits on every rank
            for a, b in zip(o[:4] + (o[4].ws,), outs[0][:4] + (es.ws,)):
                assert torch.equal(_bytes(a), _bytes(b))
        # the local kernel on the rank-summed buffer: same centres, same E-step workspace byte for byte
        ms = kmeans._MStep(1, d, k, 'cuda')
        ms.sums, ms.counts = s_ref.cuda(), counts.sum(0).int().cuda()
        es_local = kmeans._EStep(k, d, 'cuda')
        es_local.ws.zero_()
        c_local = torch.empty(k, d, device='cuda')
        ms.finalize(None, c_local, estep=es_local)
        assert torch.equal(c_local.view(torch.int32), c_new.view(torch.int32))
        assert torch.equal(es_local.ws, es.ws)
        if _lib.load().scd_estep_uses_tensor_cores(1, d, k):            # the E-step's own centroid split of c_new
            es_own = kmeans._EStep(k, d, 'cuda')
            es_own.run(torch.zeros(1, d, device='cuda'), c_new, torch.empty(1, dtype=torch.int64, device='cuda'), None)
            for a, b in zip(_es_planes(es_own.ws, k, d), _es_planes(es.ws, k, d)):
                assert torch.equal(a, b)
        hi, lo = (t.view(torch.bfloat16).view(k, d).float() for t in _es_planes(es.ws, k, d)[:2])
        assert _bits_equal(hi, c_ref.bfloat16().float()) and _bits_equal(lo, (c_ref - c_ref.bfloat16().float()).bfloat16().float())
    # null optional outputs (no C_old, move norms, counts, inertia or E-step workspace)
    c_bare = torch.empty(k, d, device='cuda')
    rk.launch(0, peer.MSTEP_CHANNEL, lambda: rk.px[0].finalize(rk.px[0]._blocks[1], None, c_bare, None, None, None))
    assert torch.equal(c_bare.view(torch.int32), c_new.view(torch.int32))


def test_finalize_centers_peer_replays_in_a_cuda_graph():
    """One virtual rank's finalize captured in a CUDA graph: each replay advances the device-side epoch (1, 2, 3) and gives
    the eager launch's outputs; scd_peer_barrier on its own channel keeps the protocol too."""
    world, k, d = 4, 37, 6
    g = torch.Generator().manual_seed(5)
    rk = Ranks(world, k, d)
    sums, counts, inertia = _mstep_blocks(world, k, d, g)
    for r in range(world):
        blk = rk.px[r].next_mstep_block()
        blk[0].copy_(sums[r])
        blk[1].copy_(counts[r])
        blk[2].fill_(float(inertia[r]))
    c_old = torch.randn(k, d, generator=g).cuda()
    eager = _run_finalize(rk, world, k, d, 0, c_old)[1]                      # ranks 0 .. 3 eagerly: epochs 1
    rk2 = Ranks(world, k, d)
    for r in range(world):
        rk2.px[r]._blocks[0][0].copy_(sums[r])
        rk2.px[r]._blocks[0][1].copy_(counts[r])
        rk2.px[r]._blocks[0][2].fill_(float(inertia[r]))
    px = rk2.px[1]
    c_new, norms = torch.empty(k, d, device='cuda'), torch.empty(k, device='cuda')
    cnt, inert = torch.empty(k, device='cuda'), torch.empty(1, dtype=torch.float64, device='cuda')
    es = kmeans._EStep(k, d, 'cuda')
    es.ws.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        px.finalize(px._blocks[0], c_old, c_new, norms, cnt, inert, es)
    assert int(rk2.pads()[1, peer.MSTEP_CHANNEL, EPOCH]) == 0              # capturing launched nothing
    for epoch in (1, 2, 3):
        for t in (c_new, norms, cnt, inert):                                # every output must be written again
            t.fill_(-1.0)
        es.ws.fill_(SENTINEL)
        rk2.launch(1, peer.MSTEP_CHANNEL, graph.replay)
        assert int(rk2.pads()[1, peer.MSTEP_CHANNEL, EPOCH]) == epoch
        for a, b in zip((c_new, norms, cnt, inert) + _es_planes(es.ws, k, d), eager[:4] + _es_planes(eager[4].ws, k, d)):
            assert torch.equal(_bytes(a), _bytes(b))
    for r in (0, 3, 1):
        rk2.launch(r, 7, lambda: rk2.px[r].barrier(7))


# ------------------------------------------------------------------------------------------------ E: one sharded round
def _round_data(kind, n, k, d):
    if kind == 'grid':
        g = torch.Generator(device='cuda').manual_seed(n + k)
        C0 = _sparse_rows(k, d, g)
        X, _ = _rows_near(C0, n, g)
        _assert_on_grid(X)
        _assert_on_grid(C0)
        idx = _names(n, 5, 3000, torch.Generator().manual_seed(n)).cuda()
        return X.contiguous(), C0.contiguous(), idx
    data = synth.make(synth.Config('ex', n, k, 3000, 9), d=d)
    _, idx = naming.score_topk(data['Xc'], data['W'], k=5)
    return data['X'].cuda(), data['C0'].cuda(), idx


@pytest.mark.parametrize('kind', ['grid', 'synth'])
@pytest.mark.parametrize('world', [2, 4, 8])
def test_sharded_round_through_the_product_code(world, kind):
    """Each virtual rank does what bench.py's Round does for its shard - bind_peer, zero the inertia, E-step, sums_counts,
    finalize_peer, sharded_vote(presorted=) - and the result is the single-rank round's: centres bitwise on the two-plane
    grid (every M-step sum exact in any order; 1e-5 on synth data) and the same on every rank, inertia exact on the grid,
    the vote bit for bit."""
    n, k, d = 9001, 40, 72
    X, C0, idx = _round_data(kind, n, k, d)
    # the single-rank round
    lab1 = torch.empty(n, dtype=torch.int64, device='cuda')
    inert1 = torch.zeros(1, dtype=torch.float64, device='cuda')
    kmeans._EStep(k, d, 'cuda').run(X, C0, lab1, inert1)
    ms1 = kmeans._MStep(n, d, k, 'cuda')
    ms1.sums_counts(X, lab1)
    c1 = torch.empty(k, d, device='cuda')
    ms1.finalize(C0, c1)
    want = [t.clone().cpu() for t in naming.vote_device(idx, lab1, k, 5, M)[:4]]
    # the sharded round
    rk = Ranks(world, k, d, n_total=n, k_used=5)
    st = []
    for r in range(world):
        lo, hi = sdist.shard_bounds(n, world, r)
        px, Xs = rk.px[r], X[lo:hi].clone()
        ms, es, es_next = kmeans._MStep(hi - lo, d, k, 'cuda'), kmeans._EStep(k, d, 'cuda'), kmeans._EStep(k, d, 'cuda')
        lab = torch.empty(hi - lo, dtype=torch.int64, device='cuda')
        ms.bind_peer(px, px.next_mstep_block())
        inertia = ms.peer[1][2]
        inertia.zero_()
        es.run(Xs, C0, lab, inertia)
        ms.sums_counts(Xs, lab)
        st.append((px, ms, es_next, lab, idx[lo:hi].contiguous(), torch.empty(k, d, device='cuda'),
                   torch.zeros(1, dtype=torch.float64, device='cuda')))
    for r, (px, ms, es_next, lab, _, c_new, inert) in enumerate(st):
        rk.launch(r, peer.MSTEP_CHANNEL, lambda: ms.finalize_peer(C0, c_new, inert, estep=es_next if ms.tc else None))
    # the vote: every rank's stores must have landed before any rank votes, so ranks 0 .. G-2 only exchange here and
    # vote below; the last rank runs the whole of sharded_vote
    recs = []
    for r, (px, ms, _, lab, idx_r, _, _) in enumerate(st[:-1]):
        recs.append(rk.launch(r, peer.RECORD_CHANNEL, lambda: px.gather_sorted_records(ms, idx_r, 5)))
    px, ms, _, lab, idx_r, _, _ = st[-1]
    votes = [None] * (world - 1) + [rk.launch(world - 1, peer.RECORD_CHANNEL,
                                              lambda: sdist.sharded_vote(lab, idx_r, 5, k, M, px, presorted=ms))]
    for r in range(world - 1):
        votes[r] = naming.vote_segments(*recs[r], k, M, n_total=n)
    for r in range(world):
        lo, hi = sdist.shard_bounds(n, world, r)
        assert torch.equal(st[r][3], lab1[lo:hi])
        c_new, inert = st[r][5], st[r][6]
        assert torch.equal(c_new.view(torch.int32), st[0][5].view(torch.int32))
        if kind == 'grid':
            assert torch.equal(c_new.view(torch.int32), c1.view(torch.int32))
            assert torch.equal(inert, inert1)
        else:
            assert torch.allclose(c_new, c1, atol=1e-5, rtol=1e-5, equal_nan=True)
            assert abs(float(inert) - float(inert1)) <= 1e-9 * float(inert1)
        names, counts, distinct, rows, ovf = votes[r]
        assert int(ovf.item()) == 0
        for a, b in zip((names, counts, distinct, rows), want):
            assert torch.equal(a.cpu(), b)
