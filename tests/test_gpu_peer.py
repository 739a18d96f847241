"""Two ranks on two GPUs (skipped on a single-GPU box): the exchange steps over NVLink peer memory - the fused
all-reduce + divide of the M-step (scd_finalize_centers_peer) and the vote records stored into every rank
(scd_pack_vote_records_peer + scd_peer_barrier) - against the NCCL path and against the single-rank result."""
import os
import socket
import traceback

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, errq):
    try:
        import datetime
        import torch.distributed as dist
        os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
        torch.cuda.set_device(rank)
        dist.init_process_group('nccl', rank=rank, world_size=world, timeout=datetime.timedelta(seconds=180),
                                device_id=torch.device('cuda', rank))
        from scd_b200 import dist as sdist, kmeans, naming, peer, synth
        group = dist.group.WORLD
        assert peer.available(group)
        cfg = synth.Config('peer', 9002, 24, 3000, 5)
        data = synth.make(cfg, d=256)
        X, Xc, W = data['X'], data['Xc'], data['W']
        lo, hi = sdist.shard_bounds(cfg.n, world, rank)
        Xs = X[lo:hi].cuda()

        # ---- fit over peer memory == fit over NCCL (same reduction order for G = 2) == single-rank fit within rounding
        one = kmeans.K_Means(k=cfg.k, max_iterations=6, n_init=1, init='random', random_state=7)
        one.fit(X.cuda())
        fits = {}
        for ex in ('peer', 'nccl'):
            os.environ['SCD_B200_EXCHANGE'] = ex
            sh = kmeans.K_Means(k=cfg.k, max_iterations=6, n_init=2, init='random', random_state=7, process_group=group)
            sh.fit(Xs)
            assert (sh._peer_exchange(cfg.k, 256, Xs.device) is not None) == (ex == 'peer')
            fits[ex] = sh
            both = [torch.empty_like(sh.cluster_centers_) for _ in range(world)]
            dist.all_gather(both, sh.cluster_centers_.contiguous())
            assert all(torch.equal(both[0].view(torch.int32), b.view(torch.int32)) for b in both[1:]), f'{ex}: centres differ between the ranks'
            assert sh.n_iter_ == one.n_iter_
            assert torch.allclose(sh.cluster_centers_, one.cluster_centers_, atol=1e-5, rtol=1e-5, equal_nan=True)
            assert (sh.labels_ == one.labels_[lo:hi]).float().mean().item() > 0.999
            assert abs(float(sh.inertia_) - float(one.inertia_)) < 1e-4 * max(1.0, float(one.inertia_))
        os.environ['SCD_B200_EXCHANGE'] = 'peer'
        assert torch.allclose(fits['peer'].cluster_centers_, fits['nccl'].cluster_centers_, atol=1e-6, rtol=1e-6, equal_nan=True)
        assert (fits['peer'].labels_ == fits['nccl'].labels_).float().mean().item() > 0.999   # NCCL's reduction order may differ from rank order

        # ---- fit_mix (labelled rows replicated, counted once) and k-means++ with random_state=None over peer memory
        y = data['y']
        lab_mask = y < 6
        L, lt = X[lab_mask][:300], y[lab_mask][:300]
        U = X[~lab_mask]
        ulo, uhi = sdist.shard_bounds(len(U), world, rank)
        one = kmeans.K_Means(k=6, max_iterations=5, n_init=1, random_state=1)
        one.fit_mix(U.cuda(), L.cuda(), lt.cuda())
        sh = kmeans.K_Means(k=6, max_iterations=5, n_init=1, random_state=1, process_group=group)
        sh.fit_mix(U[ulo:uhi].cuda(), L.cuda(), lt.cuda())
        assert torch.allclose(sh.cluster_centers_, one.cluster_centers_, atol=1e-5, rtol=1e-5)
        assert sh.n_iter_ == one.n_iter_ == len(lt)
        sh = kmeans.K_Means(k=12, max_iterations=4, n_init=2, random_state=None, process_group=group)
        sh.fit_mix(U[ulo:uhi].cuda(), L.cuda(), lt.cuda())
        both = [torch.empty_like(sh.cluster_centers_) for _ in range(world)]
        dist.all_gather(both, sh.cluster_centers_.contiguous())
        assert all(torch.equal(both[0].view(torch.int32), b.view(torch.int32)) for b in both[1:])

        # ---- a width that is not a multiple of 4 (scalar peer loads, fp32 direct-form E-step)
        g6 = torch.Generator().manual_seed(3)
        X6 = torch.randn(2000, 6, generator=g6) + 3.0 * torch.randn(5, 6, generator=g6)[torch.randint(0, 5, (2000,), generator=g6)]
        l6, h6 = sdist.shard_bounds(2000, world, rank)
        one = kmeans.K_Means(k=5, max_iterations=8, n_init=1, init='first')
        one.fit(X6.cuda())
        sh = kmeans.K_Means(k=5, max_iterations=8, n_init=1, init='first', process_group=group)
        sh.fit(X6[l6:h6].cuda())
        assert sh._peer_exchange(5, 6, torch.device('cuda', rank)) is not None
        assert torch.allclose(sh.cluster_centers_, one.cluster_centers_, atol=1e-4, rtol=1e-4)
        assert (sh.labels_ == one.labels_[l6:h6]).float().mean().item() > 0.995

        # ---- the row-sharded round: records pushed over peer memory, vote == the single-rank vote, several rounds
        # back to back (double-buffered record arrays, device-side epochs)
        C0 = data['C0'].cuda()
        lab1 = torch.empty(cfg.n, dtype=torch.int64, device='cuda')
        kmeans._estep(X.cuda(), C0, lab1, None)
        vocab = naming.Vocabulary(W.cuda())
        _, idx1 = naming.score_topk(Xc, vocab, k=5)
        names1, counts1, distinct1, rows1, _ = naming.vote_device(idx1, lab1, cfg.k, 5, 20)
        names1, counts1, distinct1, rows1 = names1.clone(), counts1.clone(), distinct1.clone(), rows1.clone()
        lab_s, idx_s = lab1[lo:hi].contiguous(), idx1[lo:hi].contiguous()
        px = peer.PeerExchange(group, cfg.k, 256, n_total=cfg.n, k_used=5)
        for rnd in range(5):
            names, counts, distinct, rows, ovf = sdist.sharded_vote(lab_s, idx_s, 5, cfg.k, 20, px)
            assert int(ovf.item()) == 0
            assert torch.equal(names, names1) and torch.equal(counts, counts1) and torch.equal(distinct, distinct1) and torch.equal(rows, rows1)
            rec = px._records[px._rec_parity ^ 1][0][:cfg.n]
            assert torch.equal(rec[:, 0].long(), lab1) and torch.equal(rec[:, 1:].long(), idx1)
        # ---- the same vote WITHOUT sorting the gathered records: each rank sends its rows in the label-sorted order of its own
        # M-step + its offsets, every cluster is then `world` sorted runs (scd_pack_sorted_records_peer + scd_vote_segments)
        ms = kmeans._MStep(hi - lo, 256, cfg.k, torch.device('cuda', rank))
        for rnd in range(4):
            ms.sums_counts(Xs, lab_s)
            names, counts, distinct, rows, ovf = sdist.sharded_vote(lab_s, idx_s, 5, cfg.k, 20, px, presorted=ms)
            assert int(ovf.item()) == 0
            assert torch.equal(names, names1) and torch.equal(counts, counts1) and torch.equal(distinct, distinct1) and torch.equal(rows, rows1)
        rec, base, seg, sbase = px._records[px._rec_parity ^ 1]
        lab_u, idx_u = px.unpack_sorted(rec, seg)
        assert torch.equal(lab_u, lab1) and torch.equal(idx_u, idx1)
        # excluded names (the partially supervised driver drops the labelled classes' names, main_ptsup.py:638)
        known = [int(x) for x in idx1[:50, 0].unique()[:7]]
        n2, c2, d2, r2, _ = naming.vote_device(idx1, lab1, cfg.k, 5, 20, known_name_idx=known)
        n2, c2 = n2.clone(), c2.clone()
        ms.sums_counts(Xs, lab_s)
        names, counts, _, _, _ = sdist.sharded_vote(lab_s, idx_s, 5, cfg.k, 20, px, presorted=ms, known_name_idx=known)
        assert torch.equal(names, n2) and torch.equal(counts, c2)
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)
    except Exception:
        errq.put(f'rank {rank}:\n{traceback.format_exc()}')
        raise


@pytest.mark.timeout(600)
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_peer_exchange_on_two_gpus():
    """World size 2, or SCD_PEER_TEST_WORLD (<= the GPUs of the box; run once at 8 - profiles/r2z_peer_test_world8.txt)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    errq = ctx.SimpleQueue()
    port = _free_port()
    world = max(2, min(int(os.environ.get('SCD_PEER_TEST_WORLD', '2')), torch.cuda.device_count()))
    procs = [ctx.Process(target=_worker, args=(r, world, port, errq)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(570)
    msgs = []
    while not errq.empty():
        msgs.append(errq.get())
    alive = [p for p in procs if p.is_alive()]
    for p in alive:
        p.kill()
    assert not msgs, '\n'.join(msgs)
    assert not alive, 'a rank did not finish'
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
